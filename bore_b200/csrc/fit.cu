// K1: fused classifier training (sm_100a, FP32 FFMA) -- the whole Keras `fit` in one launch.
//
// Replaces keras Model.fit(X, z, epochs, batch_size, shuffle=True) with optimizer="adam" and
// binary cross-entropy (README.rst:66,93; bore/plugins/hpbandster/base.py:156-157,184), which
// in the reference is epochs*ceil(N/B) TensorFlow dispatches of ~20 tiny ops each.
//
// One CTA per model; grid = number of models trained concurrently (seeds / BO problems /
// per-budget classifiers).  Per minibatch step, entirely inside the CTA:
//   gather   rows perm[e][s*B .. ) of X into shared memory, transposed to [feature][sample]
//   forward  Dense layers as register-tiled (4 samples x 4 units per thread) FFMA GEMMs on
//            shared-memory weights; activations kept for the reverse pass
//   loss     sigmoid_cross_entropy_with_logits on the final pre-activation (both Keras forms,
//            see oracle/keras_mlp.py:bce_with_logits), mean over the batch (+ l2 terms)
//   reverse  delta_{l-1} = (delta_l W_l^T) . act'(h_{l-1}) on a transposed copy of the weights
//   update   dW_l = h_{l-1}^T delta_l accumulated in registers by the thread that owns the
//            weight, Adam applied in place (Keras form: eps outside the bias correction),
//            both weight layouts rewritten; Adam slots m, v stream through L2.
// Weights never leave shared memory during the run; HBM traffic is the minibatch gather
// (B*(D+1)*4 bytes per step) plus the per-epoch loss.
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "common.cuh"
#include "fit_common.cuh"

namespace {

constexpr int FIT_THREADS = 256;

struct FitPlan {
  int w[BORE_MAX_LAYERS];    // W_l  [in][JP]          (all Dense layers incl. final)
  int wt[BORE_MAX_LAYERS];   // W_l^T [out][KP]        (layers 1.. only: layer 0 needs no reverse)
  int b[BORE_MAX_LAYERS];    // bias [JP]
  int JP[BORE_MAX_LAYERS], KP[BORE_MAX_LAYERS];  // leading dimensions of W_l / W_l^T
  int ks[BORE_MAX_LAYERS];   // sample-split of layer l's weight-gradient pass (0: the tile owner
                             // applies Adam straight from registers, no scratch)
  int h[BORE_MAX_LAYERS + 1];// activations [dim][BS]; h[0] = input batch
  int dl[2];                 // delta ping/pong [maxw][BS]
  int zb;                    // labels [BS]
  int red;                   // reduction scratch [32]
  int idx;                   // gathered row indices [BS] (ints)
  int nk[BORE_MAX_LAYERS], nj[BORE_MAX_LAYERS];  // narrow register tile (rows k x columns j) of layer l's
                             // weight-gradient pass when 4 x 4 tiles would leave threads idle (0: not used)
  int gs;                    // gradient partials [ks][in*out + out] of the layer in flight
  int total;                 // floats
  int BS;
};

__host__ __device__ inline int r4(int a) { return (a + 3) & ~3; }

// `threads`: CTA size the plan is made for (the sample-split of the gradient passes spreads
// each layer's tiles over all of them); smem_limit: floats available, splits are dropped if the
// gradient scratch does not fit
__host__ __device__ inline void make_fit_plan(const MlpDesc &d, int batch, int threads, int smem_limit,
                                              FitPlan &p, int narrow = 1) {
  const int L = d.n_layers;
  int BS = r4(batch) + 4;
  p.BS = BS;
  int off = 0, maxw = 1;
  for (int l = 0; l < L; ++l) {
    const int in = d.dims[l], out = d.dims[l + 1];
    p.JP[l] = r4(out);
    p.KP[l] = r4(in) + 4;  // +4: the Adam pass writes W^T with consecutive j (stride KP) per lane
    p.w[l] = off; off += in * p.JP[l];
    p.b[l] = off; off += p.JP[l];
    p.wt[l] = off; if (l > 0) off += out * p.KP[l];
    if (out > maxw) maxw = out;
  }
  for (int l = 0; l <= L; ++l) { p.h[l] = off; off += d.dims[l] * BS; }
  p.dl[0] = off; off += maxw * BS;
  p.dl[1] = off; off += maxw * BS;
  p.zb = off; off += BS;
  p.red = off; off += 32;
  p.idx = off; off += BS;
  // sample-split per layer: as many splits (power of two) as leave every thread at most one
  // partial tile, each split at least one 4-sample chunk
  const int nchunk = r4(batch) / 4;
  int gmax = 0;
  for (int l = 0; l < L; ++l) {
    const int in = d.dims[l], out = d.dims[l + 1];
    const int items = out == 1 ? in : ((in + 3) / 4) * (p.JP[l] / 4);
    int ks = 1;
    while (items * ks * 2 <= threads && ks * 2 <= nchunk && ks < 16) ks *= 2;
    if (out > 1 && ks == 1) ks = 0;  // enough tiles already: direct path
    p.nk[l] = p.nj[l] = 0;
    if (out > 1 && ks >= 2 && narrow) {
      // fewer 4 x 4 tiles than threads: instead of splitting the tiles over the samples (partials through
      // shared memory, summed again by the Adam pass -- 14 % of the kernel's instructions at Dense32 sizes)
      // give every thread ONE smaller tile over all samples; its owner applies Adam from registers.
      // The smallest shape that still has at most one tile per thread.
      const int shapes[4][2] = {{1, 1}, {2, 1}, {2, 2}, {4, 2}};
      for (int q = 0; q < 4; ++q) {
        const int tk = shapes[q][0], tj = shapes[q][1];
        if (((in + tk - 1) / tk) * ((out + tj - 1) / tj) <= threads) { p.nk[l] = tk; p.nj[l] = tj; break; }
      }
      if (p.nk[l]) ks = 0;
    }
    p.ks[l] = ks;
    const int need = ks * (in * out + out);
    if (need > gmax) gmax = need;
  }
  if (off + r4(gmax) > smem_limit) {  // big nets: keep only the (tiny) scratch of 1-unit layers
    gmax = 0;
    for (int l = 0; l < L; ++l) {
      const int in = d.dims[l], out = d.dims[l + 1];
      if (out > 1) p.ks[l] = 0;
      const int need = p.ks[l] * (in * out + out);
      if (need > gmax) gmax = need;
    }
  }
  p.gs = off; off += r4(gmax);
  p.total = r4(off);
}

struct FitArgs {
  MlpDesc d;
  FitPlan P;
  float *params, *adam_m, *adam_v;
  long long *adam_t;
  int model0;
  const float *X, *z;
  int N, shared_data, batch, epochs;
  const int *perm;
  int shared_perm;
  float l2k[BORE_MAX_LAYERS], l2b[BORE_MAX_LAYERS];
  int any_l2;
  float *loss_out;
  OptHyper opt;
  FitWeights fw;
  const FitProblem *probs;  // NULL: uniform launch
  float *opt_cache;         // [n_models] Nadam's momentum cache
};

// acc[i][u] += sum_k A[k*lda + i] * B[k*ldb + u]: the 4 x 4 register tile of every GEMM below
__device__ __forceinline__ void tile_fma(const float *__restrict__ ap, int lda, const float *__restrict__ bp,
                                         int ldb, int K, float (&acc)[4][4]) {
#pragma unroll 4
  for (int k = 0; k < K; ++k) {
    const float4 av = *reinterpret_cast<const float4 *>(ap + k * lda);
    const float4 wv = *reinterpret_cast<const float4 *>(bp + k * ldb);
    const float a4[4] = {av.x, av.y, av.z, av.w};
    const float w4[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int u = 0; u < 4; ++u) acc[i][u] = fmaf(a4[i], w4[u], acc[i][u]);
  }
}

// One narrow weight-gradient tile over all samples: acc[i][u] = sum_p Hin[k_i][p] DL[j_u][p], k_i = k0 + i
// (adjacent rows), j_u = j0 + u * jstep (strided: consecutive lanes own consecutive columns, so the delta
// rows of a warp are consecutive -- conflict-free float4 loads -- and its Adam-slot traffic is coalesced).
template <int TK, int TJ>
__device__ __forceinline__ void narrow_tile(const float *__restrict__ Hin, const float *__restrict__ DL, int BS,
                                            int BP, int k0, int in, int j0, int jstep, int out,
                                            float (&acc)[8]) {
  const float *hp[TK], *dp[TJ];
#pragma unroll
  for (int i = 0; i < TK; ++i) hp[i] = Hin + min(k0 + i, in - 1) * BS;
#pragma unroll
  for (int u = 0; u < TJ; ++u) dp[u] = DL + min(j0 + u * jstep, out - 1) * BS;
#pragma unroll
  for (int q = 0; q < 8; ++q) acc[q] = 0.f;
#pragma unroll 2
  for (int p = 0; p < BP; p += 4) {
    float4 hv[TK], dv[TJ];
#pragma unroll
    for (int i = 0; i < TK; ++i) hv[i] = *reinterpret_cast<const float4 *>(hp[i] + p);
#pragma unroll
    for (int u = 0; u < TJ; ++u) dv[u] = *reinterpret_cast<const float4 *>(dp[u] + p);
#pragma unroll
    for (int i = 0; i < TK; ++i)
#pragma unroll
      for (int u = 0; u < TJ; ++u) {
        float c = acc[i * TJ + u];
        c = fmaf(hv[i].x, dv[u].x, c);
        c = fmaf(hv[i].y, dv[u].y, c);
        c = fmaf(hv[i].z, dv[u].z, c);
        c = fmaf(hv[i].w, dv[u].w, c);
        acc[i * TJ + u] = c;
      }
  }
}

// Phases of one minibatch step (all inside the CTA, barrier between phases):
//   gather | forward l = 0..L-1 | loss, dL/dlogit | for l = L-1..0: { delta_{l-1} AND the partial
//   weight gradients of layer l, side by side } , { Adam on layer l }.
// Every phase spreads its work over ALL threads: a layer's gradient tiles are split over the
// sample dimension (FitPlan::ks) until there is one partial tile per thread, the partials meet
// in a shared-memory scratch, and the Adam pass walks the layer's parameters one per thread in
// flat (Keras) order, so its Adam-slot traffic is coalesced.  1-unit layers (the output layer)
// use dot-product forms instead of 4x4 tiles padded with zeros.  (The first version gave every
// 4x4 gradient tile to one thread: with Dense32 layers 64 / 16 / 8 of 128 threads worked while
// the rest waited at the barrier -- 44 % of all stall samples, profiles/r01_notes.md.)
// WEIGHTED: per-sample loss weights (FitArgs::fw); the unweighted build runs none of their code.
// RAGGED: the problems come from the table FitArgs::probs (bore_mlp_fit_ragged); the uniform build keeps the
// expressions of before: deriving its problem through fit_problem() cost cfg 4 0.4 % (132.0 -> 132.5 ms)
// EXT: the activation codes above BORE_ACT_TANH (act.cuh).  OPT: the optimizers other than Adam (opt.cuh).
template <bool WEIGHTED, bool RAGGED, bool EXT, bool OPT>
__global__ void __launch_bounds__(FIT_THREADS, 2) fit_kernel(const FitArgs a) {
  extern __shared__ __align__(16) float sm[];
  const MlpDesc &d = a.d;
  const FitPlan &P = a.P;
  const int L = d.n_layers, BS = P.BS;
  const int tid = threadIdx.x, NT = blockDim.x;
  // this CTA's problem: from the table (ragged), else the expressions of the uniform launch
  const FitProblem pb = RAGGED ? a.probs[blockIdx.x] : FitProblem{};
  const int model = RAGGED ? pb.model : a.model0 + blockIdx.x;
  const int N = RAGGED ? pb.N : a.N, epochs = RAGGED ? pb.epochs : a.epochs;
  const size_t row0 = RAGGED ? (size_t)pb.row0 : (a.shared_data ? 0 : (size_t)blockIdx.x * a.N);
  float *gp = a.params + (size_t)model * d.n_params;
  float *gm = a.adam_m + (size_t)model * d.n_params;
  float *gv = a.adam_v + (size_t)model * d.n_params;
  const float *X = a.X + (RAGGED ? (size_t)pb.row0 * d.dims[0]
                                 : (a.shared_data ? 0 : (size_t)blockIdx.x * a.N * d.dims[0]));
  const float *zg = a.z + row0;
  const int *perm = a.perm + (RAGGED ? (size_t)pb.perm0 : (a.shared_perm ? 0 : (size_t)blockIdx.x * a.epochs * a.N));
  const float *wg = WEIGHTED && a.fw.w ? a.fw.w + row0 : nullptr;
  int *idxb = reinterpret_cast<int *>(sm + P.idx);
  float *red = sm + P.red;
  float *gs = sm + P.gs;
  // loss weights of the minibatch (weighted fits): delta buffer 1 is first written by the reverse pass,
  // after the loss has read them, and last read before the barrier that ends the previous step
  float *wsm = sm + P.dl[1];
  const int D = d.dims[0];

  // ---- stage the weights: W_l [in][JP], W_l^T [out][KP] (l>0), bias ----
  for (int l = 0; l < L; ++l) {
    const int in = d.dims[l], out = d.dims[l + 1], JP = P.JP[l], KP = P.KP[l];
    for (int e = tid; e < in * JP; e += NT) {
      const int k = e / JP, j = e - k * JP;
      sm[P.w[l] + e] = j < out ? gp[d.w_off[l] + k * out + j] : 0.f;
    }
    for (int e = tid; e < JP; e += NT) sm[P.b[l] + e] = e < out ? gp[d.b_off[l] + e] : 0.f;
    if (l > 0)
      for (int e = tid; e < out * KP; e += NT) {
        const int j = e / KP, k = e - j * KP;
        sm[P.wt[l] + e] = k < in ? gp[d.w_off[l] + k * out + j] : 0.f;
      }
  }
  OptRun<OPT> run(a.opt, a.adam_t[model], a.opt_cache + model);
  const float inv_D = 1.f / (float)D;
  __syncthreads();

  const int steps_per_epoch = (N + a.batch - 1) / a.batch;
  for (int ep = 0; ep < epochs; ++ep) {
    float epoch_tot = 0.f;
    for (int st = 0; st < steps_per_epoch; ++st) {
      const int s0 = st * a.batch;
      const int nb = min(a.batch, N - s0);
      const int BP = r4(nb), nchunk = BP >> 2;
      const float inv_nchunk = 1.f / (float)nchunk;
      // ---- gather the minibatch (transposed) ----
      for (int p = tid; p < BP; p += NT) {
        const int row = p < nb ? perm[(size_t)ep * N + s0 + p] : -1;
        idxb[p] = row;
        const float zz = row >= 0 ? zg[row] : 0.f;
        sm[P.zb + p] = zz;
        if (WEIGHTED) wsm[p] = row >= 0 ? fit_sample_weight(a.fw, wg, row, zz) : 0.f;
      }
      __syncthreads();
      for (int e = tid; e < BP * D; e += NT) {
        const int p = fdiv(e, inv_D), k = e - p * D;
        const int row = idxb[p];
        sm[P.h[0] + k * BS + p] = row >= 0 ? X[(size_t)row * D + k] : 0.f;
      }
      __syncthreads();

      // ---- forward ----
      for (int l = 0; l < L; ++l) {
        const int in = d.dims[l], out = d.dims[l + 1], JP = P.JP[l];
        const float *A = sm + P.h[l];
        const float *W = sm + P.w[l];
        const float *bs = sm + P.b[l];
        float *H = sm + P.h[l + 1];
        const int act = (l == L - 1) ? BORE_ACT_LINEAR : d.act[l];  // loss works on the logit
        if (out == 1) {
          // u[p] = b + sum_k h[k][p] w[k]: one 4-sample chunk per group of kf adjacent lanes,
          // k interleaved over the group, partial sums combined by shuffle
          int kf = 1;
          while (kf < 8 && nchunk * kf * 2 <= NT) kf *= 2;
          const int per_pass = NT / kf;
          for (int base = 0; base < nchunk; base += per_pass) {
            const int c = base + tid / kf, s = tid & (kf - 1);
            const bool valid = c < nchunk;
            const float *ap = A + 4 * (valid ? c : 0);
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int k = s; k < in; k += kf) {
              const float4 av = *reinterpret_cast<const float4 *>(ap + k * BS);
              const float w = W[k * JP];
              acc.x = fmaf(av.x, w, acc.x); acc.y = fmaf(av.y, w, acc.y);
              acc.z = fmaf(av.z, w, acc.z); acc.w = fmaf(av.w, w, acc.w);
            }
            for (int o = kf >> 1; o > 0; o >>= 1) {
              acc.x += __shfl_xor_sync(0xffffffffu, acc.x, o);
              acc.y += __shfl_xor_sync(0xffffffffu, acc.y, o);
              acc.z += __shfl_xor_sync(0xffffffffu, acc.z, o);
              acc.w += __shfl_xor_sync(0xffffffffu, acc.w, o);
            }
            if (valid && s == 0) {
              const float b = bs[0];
              *reinterpret_cast<float4 *>(H + 4 * c) = make_float4(act_fwd<EXT>(act, acc.x + b), act_fwd<EXT>(act, acc.y + b),
                                                                   act_fwd<EXT>(act, acc.z + b), act_fwd<EXT>(act, acc.w + b));
            }
          }
        } else {
          const int ntile = nchunk * (JP / 4);
          for (int tt = tid; tt < ntile; tt += NT) {
            const int tj = fdiv(tt, inv_nchunk), tp = tt - tj * nchunk;
            float acc[4][4] = {};
            tile_fma(A + tp * 4, BS, W + tj * 4, JP, in, acc);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const int j = tj * 4 + u;
              if (j < out) {
                const float b = bs[j];
                float4 o;
                o.x = act_fwd<EXT>(act, acc[0][u] + b);
                o.y = act_fwd<EXT>(act, acc[1][u] + b);
                o.z = act_fwd<EXT>(act, acc[2][u] + b);
                o.w = act_fwd<EXT>(act, acc[3][u] + b);
                *reinterpret_cast<float4 *>(H + j * BS + tp * 4) = o;
              }
            }
          }
        }
        __syncthreads();
      }

      // ---- loss and dL/dlogit (mean over the batch; weighted: sum of w_i l_i over the batch size) ----
      const float inv_nb = 1.f / (float)nb;
      float lsum = 0.f;
      {
        const float *U = sm + P.h[L];  // [1][BS] logits
        float *dz = sm + P.dl[0];
        for (int p = tid; p < BP; p += NT) {
          float dl = 0.f;
          if (p < nb) {
            const float u = U[p], zz = sm[P.zb + p];
            float l = fmaxf(u, 0.f) - u * zz + log1pf(expf(-fabsf(u))), g = stable_sigmoid(u) - zz;
            if (WEIGHTED) { const float ws = wsm[p]; l *= ws; g *= ws; }
            lsum += l;
            dl = g * inv_nb;
          }
          dz[p] = dl;
        }
      }
      float loss = block_sum(lsum, red) * inv_nb;  // (also the barrier publishing dz)

      // ---- optimizer scalars for this step ----
      const OptStep os = run.step(a.opt);
      float reg = 0.f;

      // ---- reverse + update, top layer first ----
      int cur = 0;
      for (int l = L - 1; l >= 0; --l) {
        const int in = d.dims[l], out = d.dims[l + 1], JP = P.JP[l], KP = P.KP[l];
        const float inv_out = 1.f / (float)out;
        const float *DL = sm + P.dl[cur];  // delta_l [out][BS]
        const float *Hin = sm + P.h[l];    // input of layer l = output of layer l-1
        const int ks = P.ks[l];
        const int psz = in * out + out;    // layer l's parameters, flat: W_l then b_l
        // (1) delta_{l-1} = (delta_l W_l^T) . act'(h_{l-1}) into the other buffer
        if (l > 0) {
          const float *WT = sm + P.wt[l];
          float *DN = sm + P.dl[cur ^ 1];
          const int actp = d.act[l - 1];
          if (out == 1) {
            for (int e = tid; e < in * nchunk; e += NT) {
              const int k = fdiv(e, inv_nchunk), c = e - k * nchunk;
              const float4 dv = *reinterpret_cast<const float4 *>(DL + 4 * c);
              const float4 hv = *reinterpret_cast<const float4 *>(Hin + k * BS + 4 * c);
              const float w = WT[k];
              *reinterpret_cast<float4 *>(DN + k * BS + 4 * c) =
                  make_float4(dv.x * w * act_bwd<EXT>(actp, hv.x), dv.y * w * act_bwd<EXT>(actp, hv.y),
                              dv.z * w * act_bwd<EXT>(actp, hv.z), dv.w * w * act_bwd<EXT>(actp, hv.w));
            }
          } else {
            const int ntile = nchunk * (r4(in) / 4);
            for (int tt = tid; tt < ntile; tt += NT) {
              const int tk = fdiv(tt, inv_nchunk), tp = tt - tk * nchunk;
              float acc[4][4] = {};
              tile_fma(DL + tp * 4, BS, WT + tk * 4, KP, out, acc);
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                const int k = tk * 4 + u;
                if (k < in) {
                  const float4 hv = *reinterpret_cast<const float4 *>(Hin + k * BS + tp * 4);
                  float4 o;
                  o.x = acc[0][u] * act_bwd<EXT>(actp, hv.x);
                  o.y = acc[1][u] * act_bwd<EXT>(actp, hv.y);
                  o.z = acc[2][u] * act_bwd<EXT>(actp, hv.z);
                  o.w = acc[3][u] * act_bwd<EXT>(actp, hv.w);
                  *reinterpret_cast<float4 *>(DN + k * BS + tp * 4) = o;
                }
              }
            }
          }
        }
        if (P.nk[l] > 0) {
          // (2n) one narrow register tile per thread over ALL samples, in the same phase as (1) (both only
          //      read); after ONE barrier its owner applies Adam straight from registers.  No trailing
          //      barrier: the next layer's phase reads delta_{l-1} (complete before this barrier) and
          //      weights that nobody is writing.
          const int TK = P.nk[l], TJ = P.nj[l];
          const int tjn = (out + TJ - 1) / TJ, tkn = (in + TK - 1) / TK;
          const bool has = tid < tjn * tkn;
          const int tk = has ? tid / tjn : 0, tj = has ? tid - tk * tjn : 0;
          const int k0 = tk * TK;
          float acc[8], am[8], av[8];
          if (has) {
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              am[q] = 0.f; av[q] = 0.f;
              const int i = q / TJ, u = q - i * TJ;  // (TJ is 1 or 2)
              if (q < TK * TJ) {
                const int gi = d.w_off[l] + min(k0 + i, in - 1) * out + min(tj + u * tjn, out - 1);
                am[q] = __ldcg(gm + gi);
                av[q] = __ldcg(gv + gi);
              }
            }
            if (TK == 4) narrow_tile<4, 2>(Hin, DL, BS, BP, k0, in, tj, tjn, out, acc);
            else if (TJ == 2) narrow_tile<2, 2>(Hin, DL, BS, BP, k0, in, tj, tjn, out, acc);
            else if (TK == 2) narrow_tile<2, 1>(Hin, DL, BS, BP, k0, in, tj, tjn, out, acc);
            else narrow_tile<1, 1>(Hin, DL, BS, BP, k0, in, tj, tjn, out, acc);
          }
          // bias gradient db_j = sum_p delta_l[j][p] by the LAST threads (the first ones own the tiles)
          const int jb = NT - 1 - tid;
          float gb = 0.f, bm = 0.f, bvv = 0.f;
          if (jb < out) {
            bm = __ldcg(gm + d.b_off[l] + jb);
            bvv = __ldcg(gv + d.b_off[l] + jb);
            for (int p = 0; p < BP; p += 4) {
              const float4 dv = *reinterpret_cast<const float4 *>(DL + jb * BS + p);
              gb += (dv.x + dv.y) + (dv.z + dv.w);
            }
          }
          __syncthreads();  // every read of W_l / W_l^T / delta_l of this phase is done
          {
            float *W = sm + P.w[l];
            float *WT = sm + P.wt[l];
            const float l2k = a.l2k[l], l2b = a.l2b[l];
            if (has) {
#pragma unroll
              for (int q = 0; q < 8; ++q) {
                const int i = q / TJ, u = q - i * TJ;
                const int k = k0 + i, j = tj + u * tjn;
                if (q < TK * TJ && k < in && j < out) {
                  const int gi = d.w_off[l] + k * out + j;
                  float wv = W[k * JP + j];
                  float g = acc[q];
                  if (l2k != 0.f) { reg += l2k * wv * wv; g += 2.f * l2k * wv; }
                  float m = am[q], v = av[q];
                  wv = opt_update<OPT>(a.opt, os, wv, g, m, v);
                  gm[gi] = m; gv[gi] = v;
                  W[k * JP + j] = wv;
                  if (l > 0) WT[j * KP + k] = wv;
                }
              }
            }
            if (jb < out) {
              const int gi = d.b_off[l] + jb;
              float bv = sm[P.b[l] + jb];
              if (l2b != 0.f) { reg += l2b * bv * bv; gb += 2.f * l2b * bv; }
              bv = opt_update<OPT>(a.opt, os, bv, gb, bm, bvv);
              gm[gi] = bm; gv[gi] = bvv;
              sm[P.b[l] + jb] = bv;
            }
          }
          cur ^= 1;
          continue;
        }
        if (ks > 0) {
          // (2a) partial gradients of layer l over sample split s, into gs[s][psz] -- same phase as
          //      (1): both only read.  chunks [c0, c1) of 4 samples belong to split s.
          const int cps = (nchunk + ks - 1) >> (__ffs(ks) - 1);  // ks is a power of two
          if (out == 1) {
            const float inv_in1 = 1.f / (float)(in + 1);
            for (int e = tid; e < (in + 1) * ks; e += NT) {
              const int s = fdiv(e, inv_in1), k = e - s * (in + 1);
              const int c0 = s * cps, c1 = min(c0 + cps, nchunk);
              float g = 0.f;
              for (int c = c0; c < c1; ++c) {
                const float4 dv = *reinterpret_cast<const float4 *>(DL + 4 * c);
                if (k < in) {
                  const float4 hv = *reinterpret_cast<const float4 *>(Hin + k * BS + 4 * c);
                  g = fmaf(hv.x, dv.x, g); g = fmaf(hv.y, dv.y, g);
                  g = fmaf(hv.z, dv.z, g); g = fmaf(hv.w, dv.w, g);
                } else {
                  g += (dv.x + dv.y) + (dv.z + dv.w);
                }
              }
              gs[s * psz + k] = g;  // k == in: the bias slot
            }
          } else {
            const int tjn = JP / 4, tkn = (in + 3) / 4, ntile = tkn * tjn;
            const float inv_ntile = 1.f / (float)ntile, inv_tjn = 1.f / (float)tjn;
            for (int e = tid; e < ntile * ks; e += NT) {
              const int s = fdiv(e, inv_ntile), tt = e - s * ntile;
              const int tk = fdiv(tt, inv_tjn), tj = tt - tk * tjn;
              // lanes walk j (rows tj, tj + tjn, ... of delta: bank-conflict-free float4 loads, and
              // contiguous scalar stores below); the 4 k rows of a tile are adjacent
              const int c0 = s * cps, c1 = min(c0 + cps, nchunk);
              float acc[4][4] = {};
              int kk[4], jj[4];
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                kk[u] = min(tk * 4 + u, in - 1);
                jj[u] = min(tj + u * tjn, out - 1);
              }
              for (int c = c0; c < c1; ++c) {
                float4 hv[4], dv[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                  hv[u] = *reinterpret_cast<const float4 *>(Hin + kk[u] * BS + 4 * c);
                  dv[u] = *reinterpret_cast<const float4 *>(DL + jj[u] * BS + 4 * c);
                }
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                  for (int u = 0; u < 4; ++u) {
                    acc[i][u] = fmaf(hv[i].x, dv[u].x, acc[i][u]);
                    acc[i][u] = fmaf(hv[i].y, dv[u].y, acc[i][u]);
                    acc[i][u] = fmaf(hv[i].z, dv[u].z, acc[i][u]);
                    acc[i][u] = fmaf(hv[i].w, dv[u].w, acc[i][u]);
                  }
              }
              float *gp_s = gs + s * psz;
              if (((in | out) & 3) == 0) {  // whole tiles: no predicates, one base address
                float *dp = gp_s + tk * 4 * out + tj;
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                  for (int u = 0; u < 4; ++u) dp[i * out + u * tjn] = acc[i][u];
              } else {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                  const int k = tk * 4 + i;
                  if (k >= in) continue;
#pragma unroll
                  for (int u = 0; u < 4; ++u) {
                    const int j = tj + u * tjn;
                    if (j < out) gp_s[k * out + j] = acc[i][u];
                  }
                }
              }
            }
            // bias partials: db_j over split s
            for (int e = tid; e < out * ks; e += NT) {
              const int s = fdiv(e, inv_out), j = e - s * out;
              const int c0 = s * cps, c1 = min(c0 + cps, nchunk);
              float g = 0.f;
              for (int c = c0; c < c1; ++c) {
                const float4 dv = *reinterpret_cast<const float4 *>(DL + j * BS + 4 * c);
                g += (dv.x + dv.y) + (dv.z + dv.w);
              }
              gs[s * psz + in * out + j] = g;
            }
          }
          __syncthreads();
          // (2b) Adam on layer l, one parameter per thread in flat order (coalesced slot traffic);
          //      four parameters' slots are requested before the first is used.  Weights first,
          //      then the biases (no per-element branch between the two kinds).
          {
            float *W = sm + P.w[l];
            float *WT = sm + P.wt[l];
            float *bsm = sm + P.b[l];
            const float l2k = a.l2k[l], l2b = a.l2b[l];
            const int nw = in * out, g0 = d.w_off[l];
            auto grad_sum = [&](int e) {
              float g = gs[e];
              if (ks == 2) return g + gs[psz + e];
              for (int s = 1; s < ks; ++s) g += gs[s * psz + e];
              return g;
            };
            for (int e0 = tid; e0 < nw; e0 += 4 * NT) {
              float mq[4], vq[4];
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const int e = min(e0 + q * NT, nw - 1);
                mq[q] = __ldcg(gm + g0 + e);
                vq[q] = __ldcg(gv + g0 + e);
              }
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const int e = e0 + q * NT;
                if (e >= nw) break;
                float g = grad_sum(e);
                const int k = fdiv(e, inv_out), j = e - k * out;
                float wv = W[k * JP + j];
                if (l2k != 0.f) { reg += l2k * wv * wv; g += 2.f * l2k * wv; }
                wv = opt_update<OPT>(a.opt, os, wv, g, mq[q], vq[q]);
                W[k * JP + j] = wv;
                if (l > 0) WT[j * KP + k] = wv;
                gm[g0 + e] = mq[q];
                gv[g0 + e] = vq[q];
              }
            }
            for (int j = tid; j < out; j += NT) {
              const int e = nw + j;
              float g = grad_sum(e);
              float bv = bsm[j];
              if (l2b != 0.f) { reg += l2b * bv * bv; g += 2.f * l2b * bv; }
              float m = __ldcg(gm + g0 + e), v = __ldcg(gv + g0 + e);
              bsm[j] = opt_update<OPT>(a.opt, os, bv, g, m, v);
              gm[g0 + e] = m;
              gv[g0 + e] = v;
            }
          }
        } else {
          __syncthreads();  // delta_{l-1} done with W_l before W_l changes
          // (2') enough tiles for every thread: dW_l = h_{l-1}^T delta_l (+2*l2*w) and Adam by the
          //      tile's owner; thread tile 4(k) x 4(j), k strided so that consecutive lanes read
          //      consecutive activation rows
          float *W = sm + P.w[l];
          float *WT = sm + P.wt[l];
          const float l2k = a.l2k[l], l2b = a.l2b[l];
          const int tkn = (in + 3) / 4, tjn = JP / 4;
          const int ntile = tkn * tjn;
          for (int tt = tid; tt < ntile; tt += NT) {
            const int tk = tt % tkn, tj = tt / tkn;
            float acc[4][4] = {};
            int kk[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) kk[u] = min(tk + u * tkn, in - 1);
            // Adam slots of this tile: requested from L2 now, consumed after the GEMM loop
            float am[4][4], av[4][4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                const int gi = d.w_off[l] + kk[i] * out + min(tj * 4 + u, out - 1);
                am[i][u] = __ldcg(gm + gi);
                av[i][u] = __ldcg(gv + gi);
              }
            for (int p = 0; p < BP; p += 4) {
              float4 hv[4], dv[4];
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                hv[u] = *reinterpret_cast<const float4 *>(Hin + kk[u] * BS + p);
                dv[u] = *reinterpret_cast<const float4 *>(DL + min(tj * 4 + u, out - 1) * BS + p);
              }
#pragma unroll
              for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                  acc[i][u] = fmaf(hv[i].x, dv[u].x, acc[i][u]);
                  acc[i][u] = fmaf(hv[i].y, dv[u].y, acc[i][u]);
                  acc[i][u] = fmaf(hv[i].z, dv[u].z, acc[i][u]);
                  acc[i][u] = fmaf(hv[i].w, dv[u].w, acc[i][u]);
                }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int k = tk + i * tkn;
              if (k >= in) continue;
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                const int j = tj * 4 + u;
                if (j >= out) continue;
                const int gi = d.w_off[l] + k * out + j;
                float wv = W[k * JP + j];
                float g = acc[i][u];
                if (l2k != 0.f) { reg += l2k * wv * wv; g += 2.f * l2k * wv; }
                float m = am[i][u], v = av[i][u];
                wv = opt_update<OPT>(a.opt, os, wv, g, m, v);
                gm[gi] = m; gv[gi] = v;
                W[k * JP + j] = wv;
                if (l > 0) WT[j * KP + k] = wv;
              }
            }
          }
          // bias: db_j = sum_p delta_l[j][p]
          for (int j = tid; j < out; j += NT) {
            float g = 0.f;
            for (int p = 0; p < BP; ++p) g += DL[j * BS + p];
            const int gi = d.b_off[l] + j;
            float bv = sm[P.b[l] + j];
            if (l2b != 0.f) { reg += l2b * bv * bv; g += 2.f * l2b * bv; }
            float m = gm[gi], v = gv[gi];
            bv = opt_update<OPT>(a.opt, os, bv, g, m, v);
            gm[gi] = m; gv[gi] = v;
            sm[P.b[l] + j] = bv;
          }
        }
        __syncthreads();
        cur ^= 1;
      }
      if (a.any_l2) loss += block_sum(reg, red);
      epoch_tot += loss * (float)nb;
    }
    if (tid == 0 && a.loss_out)
      a.loss_out[(RAGGED ? (size_t)pb.loss0 : (size_t)blockIdx.x * epochs) + ep] = epoch_tot / (float)N;
  }

  // ---- write the trained weights back ----
  __syncthreads();
  for (int l = 0; l < L; ++l) {
    const int in = d.dims[l], out = d.dims[l + 1], JP = P.JP[l];
    for (int e = tid; e < in * out; e += NT) {
      const int k = e / out, j = e - k * out;
      gp[d.w_off[l] + e] = sm[P.w[l] + k * JP + j];
    }
    for (int e = tid; e < out; e += NT) gp[d.b_off[l] + e] = sm[P.b[l] + e];
  }
  if (tid == 0) run.store(a.adam_t + model, a.opt_cache + model);
}

// ---------------------------------------------------------------- K1c: one model = one CLUSTER
// A single model on a single CTA is latency bound (~10^3 strictly dependent steps, each a chain
// of small GEMM tiles on one SM).  fit_cluster_kernel spreads ONE model over a thread-block
// cluster of FIT_CLUSTER CTAs (= SMs):
//   * every CTA keeps the full weights (both layouts) in its own shared memory and carries its
//     slice of the minibatch (ceil(nb / FIT_CLUSTER) samples) through forward / loss / reverse;
//     the k-loop of every output is split over 2..8 adjacent lanes (shuffle-reduced) so that all
//     256 threads share the few hundred outputs of a layer;
//   * each CTA leaves its partial gradient (its samples only) in shared memory, flat in Keras
//     parameter order; after a cluster barrier CTA r reduces parameter slice r over all CTAs
//     through distributed shared memory (float4 loads, fixed order 0..C-1: deterministic),
//     applies Adam with the slots of that slice -- which live in ITS shared memory for the whole
//     run -- and leaves the new values in place of its own partial slice;
//   * after a second cluster barrier (the next minibatch is gathered between its arrive and its
//     wait) every CTA pulls the updated slices from their owners and rewrites its W / W^T images.
// HBM sees the minibatch gather only.  Epoch losses are assembled by rank 0 from per-CTA
// partial sums (parity slots: a CTA may be one step ahead of rank 0's read).
constexpr int FIT_CLUSTER = 8;
constexpr int FIT_CTHREADS = 512;  // threads per CTA of the cluster kernel

struct FitCPlan {
  int w[BORE_MAX_LAYERS], wt[BORE_MAX_LAYERS], b[BORE_MAX_LAYERS];
  int h[BORE_MAX_LAYERS + 1];  // activations [dim][SP]
  int dl[2];                   // delta ping/pong [maxw][SP]
  int zb, red, idx;            // labels [SP], reduction scratch [32], row indices [SP]
  int dwp;                     // partial gradient, flat [FIT_CLUSTER * chunk]
  int wn;                      // updated values of this CTA's parameter slice [chunk]
  int am, av;                  // Adam slots of this CTA's parameter slice [chunk]
  int tab;                     // flat index -> (offset in W/bias image) | (offset in W^T image + 1) << 16
  int slots;                   // lsum[2], reg[2]
  int total, SP, chunk, wend;  // wend: end of the weight images (offsets must fit 16 bits)
};

// leading dimension of the weight images: = 8 (mod 32).  In dense_pass a warp reads W[k][j] for
// 4 interleaved k (the k-split of an output over adjacent lanes) x 8 adjacent j: with this stride
// the 32 addresses fall into 32 different banks (an odd stride, the first choice, separated the k
// rows of ONE column but let (k, j) and (k+1, j-1) collide: half of all shared-memory wavefronts
// of the kernel were bank conflicts, profiles/r01_ncu_fit_cluster_v5.txt)
__host__ __device__ inline int ldo(int n) { return n <= 8 ? 8 : ((n - 8 + 31) / 32) * 32 + 8; }

__host__ __device__ inline void make_fitc_plan(const MlpDesc &d, int batch, FitCPlan &p) {
  const int L = d.n_layers;
  const int SP = r4((batch + FIT_CLUSTER - 1) / FIT_CLUSTER);
  p.SP = SP;
  p.chunk = r4((d.n_params + FIT_CLUSTER - 1) / FIT_CLUSTER);
  int off = 0, maxw = d.dims[0];
  for (int l = 0; l < L; ++l) {
    const int in = d.dims[l], out = d.dims[l + 1];
    p.w[l] = off; off += in * ldo(out);
    p.b[l] = off; off += r4(out);
    p.wt[l] = off; if (l > 0) off += out * ldo(in);
    if (out > maxw) maxw = out;
  }
  off = r4(off);
  p.wend = off;
  for (int l = 0; l <= L; ++l) { p.h[l] = off; off += d.dims[l] * SP; }
  p.dl[0] = off; off += maxw * SP;
  p.dl[1] = off; off += maxw * SP;
  p.zb = off; off += SP;
  p.red = off; off += 32;
  p.idx = off; off += SP;
  p.dwp = off; off += FIT_CLUSTER * p.chunk;
  p.wn = off; off += p.chunk;
  p.am = off; off += p.chunk;
  p.av = off; off += p.chunk;
  p.tab = off; off += FIT_CLUSTER * p.chunk;
  p.slots = off; off += 4;
  p.total = r4(off);
}

struct FitCArgs {
  MlpDesc d;
  FitCPlan P;
  float *params, *adam_m, *adam_v;
  long long *adam_t;
  int model0;
  const float *X, *z;
  int N, shared_data, batch, epochs;
  const int *perm;
  int shared_perm;
  const FitProblem *probs;  // NULL: uniform launch (fit_problem)
  float l2k[BORE_MAX_LAYERS], l2b[BORE_MAX_LAYERS];
  int any_l2;
  float *loss_out;
  OptHyper opt;
  FitWeights fw;
  float *opt_cache;  // [n_models] Nadam's momentum cache
};

__device__ __forceinline__ uint32_t cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_arrive() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
}
__device__ __forceinline__ void cluster_wait() {
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// address of `p` (a pointer into this CTA's shared memory) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t dsmem_addr(const void *p, uint32_t rank) {
  uint32_t a = (uint32_t)__cvta_generic_to_shared(p), r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(rank));
  return r;
}
__device__ __forceinline__ float dsmem_ld(uint32_t addr) {
  float v;
  asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ float4 dsmem_ld4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "r"(addr)
               : "memory");
  return v;
}

// OUT(j, q) = epi( sum_k A[k][4q..4q+3] * Wm[k*ldw + j] ) for j < nout, q < SP/4.  An output is
// shared by `ks` adjacent lanes (k interleaved, partial sums combined by shuffle); `ks` is the
// largest power of two <= 8 that still leaves every thread an output.  ldw is odd (ldo).
template <class Epi>
__device__ __forceinline__ void dense_pass(const float *A, const float *Wm, int K, int ldw, int nout,
                                           int SP, Epi epi) {
  const int nq = SP >> 2, items = nout * nq, NT = blockDim.x;
  const int ksh = (items << 3) <= NT ? 3 : (items << 2) <= NT ? 2 : (items << 1) <= NT ? 1 : 0;
  const int ks = 1 << ksh;
  const int kp = threadIdx.x & (ks - 1);
  const int per_pass = NT >> ksh;
  const float inv_nout = 1.f / (float)nout;
  // pointer strides of one k-step of this lane (no multiplications inside the loop)
  const int astep = ks * SP, wstep = ks * ldw;
  const int n_it = (K - kp + ks - 1) >> ksh;
  for (int base = 0; base < items; base += per_pass) {
    const int o = base + (threadIdx.x >> ksh);
    const bool valid = o < items;
    const int oo = valid ? o : 0;
    const int q = fdiv(oo, inv_nout), j = oo - q * nout;
    const float *ap = A + 4 * q + kp * SP;
    const float *wp = Wm + j + kp * ldw;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
    for (int it = 0; it < n_it; ++it) {
      const float4 a = *reinterpret_cast<const float4 *>(ap);
      const float w = *wp;
      ap += astep;
      wp += wstep;
      acc.x = fmaf(a.x, w, acc.x);
      acc.y = fmaf(a.y, w, acc.y);
      acc.z = fmaf(a.z, w, acc.z);
      acc.w = fmaf(a.w, w, acc.w);
    }
    for (int off = ks >> 1; off > 0; off >>= 1) {
      acc.x += __shfl_xor_sync(0xffffffffu, acc.x, off);
      acc.y += __shfl_xor_sync(0xffffffffu, acc.y, off);
      acc.z += __shfl_xor_sync(0xffffffffu, acc.z, off);
      acc.w += __shfl_xor_sync(0xffffffffu, acc.w, off);
    }
    if (valid && kp == 0) epi(j, q, acc);
  }
}

// activation of four values with ONE dispatch (the switch of act_fwd per element showed up with
// 4.6 % of the cluster kernel's instructions)
template <bool EXT>
__device__ __forceinline__ float4 f_act4(int a, float4 v) {
  if (a == BORE_ACT_RELU) return make_float4(fmaxf(v.x, 0.f), fmaxf(v.y, 0.f), fmaxf(v.z, 0.f), fmaxf(v.w, 0.f));
  if (a == BORE_ACT_LINEAR) return v;
  return make_float4(act_fwd<EXT>(a, v.x), act_fwd<EXT>(a, v.y), act_fwd<EXT>(a, v.z), act_fwd<EXT>(a, v.w));
}
// acc * act'(h), four values
template <bool EXT>
__device__ __forceinline__ float4 f_act_bwd4(int a, float4 acc, float4 h) {
  if (a == BORE_ACT_RELU)
    return make_float4(h.x > 0.f ? acc.x : 0.f, h.y > 0.f ? acc.y : 0.f, h.z > 0.f ? acc.z : 0.f,
                       h.w > 0.f ? acc.w : 0.f);
  if (a == BORE_ACT_LINEAR) return acc;
  return make_float4(acc.x * act_bwd<EXT>(a, h.x), acc.y * act_bwd<EXT>(a, h.y), acc.z * act_bwd<EXT>(a, h.z),
                     acc.w * act_bwd<EXT>(a, h.w));
}

template <bool WEIGHTED, bool EXT, bool OPT>
__global__ void __cluster_dims__(FIT_CLUSTER, 1, 1) __launch_bounds__(FIT_CTHREADS)
fit_cluster_kernel(const FitCArgs a) {
  extern __shared__ __align__(16) float sm[];
  const MlpDesc &d = a.d;
  const FitCPlan &P = a.P;
  const int L = d.n_layers, SP = P.SP;
  const int tid = threadIdx.x, NT = blockDim.x;
  const int rank = (int)cluster_rank();
  const FitProblem pb = fit_problem(a, blockIdx.x / FIT_CLUSTER);  // which problem of the launch
  const int model = pb.model, N = pb.N, epochs = pb.epochs;
  float *gp = a.params + (size_t)model * d.n_params;
  float *gm = a.adam_m + (size_t)model * d.n_params;
  float *gv = a.adam_v + (size_t)model * d.n_params;
  const float *X = a.X + pb.row0 * d.dims[0];
  const float *zg = a.z + pb.row0;
  const int *perm = a.perm + pb.perm0;
  const float *wg = WEIGHTED && a.fw.w ? a.fw.w + pb.row0 : nullptr;
  int *idxb = reinterpret_cast<int *>(sm + P.idx);
  float *red = sm + P.red;
  // loss weights of this CTA's samples (weighted fits): delta buffer 1 is dead from the end of one reverse
  // pass (where the next minibatch is gathered) to the reverse pass of the next step
  float *wsm = sm + P.dl[1];
  const int D = d.dims[0];
  const int i0 = rank * P.chunk;                       // this CTA's parameter slice
  const int i1 = min(i0 + P.chunk, d.n_params);
  const int steps_per_epoch = (N + a.batch - 1) / a.batch;

  // gathers this CTA's slice of minibatch (ep, st), transposed and zero padded; ends published
  auto gather = [&](int ep, int st) {
    const int s0 = st * a.batch;
    const int nb = min(a.batch, N - s0);
    const int spc = (nb + FIT_CLUSTER - 1) / FIT_CLUSTER;
    const int p0 = rank * spc;
    const int mine = max(0, min(spc, nb - p0));
    for (int p = tid; p < SP; p += NT) {
      const int row = p < mine ? perm[(size_t)ep * N + s0 + p0 + p] : -1;
      idxb[p] = row;
      const float zz = row >= 0 ? zg[row] : 0.f;
      sm[P.zb + p] = zz;
      if (WEIGHTED) wsm[p] = row >= 0 ? fit_sample_weight(a.fw, wg, row, zz) : 0.f;
    }
    __syncthreads();
    for (int e = tid; e < SP * D; e += NT) {
      const int p = e / D, k = e - p * D;
      const int row = idxb[p];
      sm[P.h[0] + k * SP + p] = row >= 0 ? X[(size_t)row * D + k] : 0.f;
    }
    __syncthreads();
  };
  // flat parameter index -> offsets of that parameter in the W (or bias) and W^T images
  auto locate = [&](int i, int &off_w, int &off_wt, float &l2) {
    int l = 0;
    while (l + 1 < L && i >= d.w_off[l + 1]) ++l;
    const int in = d.dims[l], out = d.dims[l + 1];
    off_wt = -1;
    if (i >= d.b_off[l]) {
      off_w = P.b[l] + (i - d.b_off[l]);
      l2 = a.l2b[l];
    } else {
      const int e = i - d.w_off[l], k = e / out, j = e - k * out;
      off_w = P.w[l] + k * ldo(out) + j;
      if (l > 0) off_wt = P.wt[l] + j * ldo(in) + k;
      l2 = a.l2k[l];
    }
  };

  // ---- stage the weights (all CTAs) and this CTA's Adam slots ----
  for (int l = 0; l < L; ++l) {
    const int in = d.dims[l], out = d.dims[l + 1], JP = ldo(out), KP = ldo(in);
    for (int e = tid; e < in * JP; e += NT) {
      const int k = e / JP, j = e - k * JP;
      sm[P.w[l] + e] = j < out ? gp[d.w_off[l] + k * out + j] : 0.f;
    }
    for (int e = tid; e < r4(out); e += NT) sm[P.b[l] + e] = e < out ? gp[d.b_off[l] + e] : 0.f;
    if (l > 0)
      for (int e = tid; e < out * KP; e += NT) {
        const int j = e / KP, k = e - j * KP;
        sm[P.wt[l] + e] = k < in ? gp[d.w_off[l] + k * out + j] : 0.f;
      }
  }
  for (int i = tid; i < P.chunk; i += NT) {
    sm[P.am + i] = i0 + i < i1 ? gm[i0 + i] : 0.f;
    sm[P.av + i] = i0 + i < i1 ? gv[i0 + i] : 0.f;
  }
  int *tab = reinterpret_cast<int *>(sm + P.tab);
  for (int i = tid; i < FIT_CLUSTER * P.chunk; i += NT) {
    sm[P.dwp + i] = 0.f;
    int code = 0xffff;  // padding: no such parameter
    if (i < d.n_params) {
      int off_w, off_wt;
      float l2;
      locate(i, off_w, off_wt, l2);
      code = off_w | (off_wt + 1) << 16;
    }
    tab[i] = code;
  }
  if (tid < 4) sm[P.slots + tid] = 0.f;
  OptRun<OPT> run(a.opt, a.adam_t[model], a.opt_cache + model);
  uint32_t peer[FIT_CLUSTER];  // base of every CTA's dynamic shared memory
#pragma unroll
  for (int c = 0; c < FIT_CLUSTER; ++c) peer[c] = dsmem_addr(sm, c);
  gather(0, 0);
  cluster_arrive();
  cluster_wait();  // everybody's shared memory exists and is initialised

  const float inv_chunk = 1.f / (float)P.chunk;
  int par = 0;  // slot parity of the current step
  for (int ep = 0; ep < epochs; ++ep) {
    float epoch_tot = 0.f;
    for (int st = 0; st < steps_per_epoch; ++st, par ^= 1) {
      const int s0 = st * a.batch;
      const int nb = min(a.batch, N - s0);
      const int spc = (nb + FIT_CLUSTER - 1) / FIT_CLUSTER;  // samples per CTA
      const int mine = max(0, min(spc, nb - rank * spc));     // this CTA's samples

      // ---- forward (the minibatch slice is already in place) ----
      for (int l = 0; l < L; ++l) {
        const int in = d.dims[l], out = d.dims[l + 1];
        const float *bs = sm + P.b[l];
        float *H = sm + P.h[l + 1];
        const int act = (l == L - 1) ? BORE_ACT_LINEAR : d.act[l];  // loss works on the logit
        dense_pass(sm + P.h[l], sm + P.w[l], in, ldo(out), out, SP, [&](int j, int q, float4 acc) {
          const float b = bs[j];
          *reinterpret_cast<float4 *>(H + j * SP + 4 * q) =
              f_act4<EXT>(act, make_float4(acc.x + b, acc.y + b, acc.z + b, acc.w + b));
        });
        __syncthreads();
      }

      // ---- loss (partial sum over this CTA's samples) and dL/dlogit (mean over the batch) ----
      const float inv_nb = 1.f / (float)nb;
      float lsum = 0.f;
      {
        const float *U = sm + P.h[L];
        float *dz = sm + P.dl[0];
        for (int p = tid; p < SP; p += NT) {
          float dl = 0.f;
          if (p < mine) {
            const float u = U[p], zz = sm[P.zb + p];
            float l = fmaxf(u, 0.f) - u * zz + log1pf(expf(-fabsf(u))), g = stable_sigmoid(u) - zz;
            if (WEIGHTED) { const float ws = wsm[p]; l *= ws; g *= ws; }
            lsum += l;
            dl = g * inv_nb;
          }
          dz[p] = dl;
        }
      }
      lsum = block_sum(lsum, red);  // (also the barrier publishing dz)
      if (tid == 0) sm[P.slots + par] = lsum;

      // ---- optimizer scalars for this step ----
      const OptStep os = run.step(a.opt);

      // ---- reverse: per layer, delta_{l-1} and this CTA's partial dW_l / db_l ----
      int cur = 0;
      for (int l = L - 1; l >= 0; --l) {
        const int in = d.dims[l], out = d.dims[l + 1];
        const float *DL = sm + P.dl[cur];  // delta_l [out][SP]
        const float *Hin = sm + P.h[l];
        if (l > 0) {
          float *DN = sm + P.dl[cur ^ 1];
          const int actp = d.act[l - 1];
          dense_pass(DL, sm + P.wt[l], out, ldo(in), in, SP, [&](int k, int q, float4 acc) {
            const float4 hv = *reinterpret_cast<const float4 *>(Hin + k * SP + 4 * q);
            *reinterpret_cast<float4 *>(DN + k * SP + 4 * q) = f_act_bwd4<EXT>(actp, acc, hv);
          });
        }
        {
          // partial dW_l = h_{l-1}^T delta_l over this CTA's samples: 4(k) x 4(j) register tiles;
          // lanes walk j (rows tj, tj + tjn, ... of delta), so the stores below are contiguous
          float *dW = sm + P.dwp + d.w_off[l];
          const int tkn = (in + 3) / 4, tjn = (out + 3) / 4;
          const float inv_tjn = 1.f / (float)tjn;
          for (int tt = tid; tt < tkn * tjn; tt += NT) {
            const int tk = fdiv(tt, inv_tjn), tj = tt - tk * tjn;
            float acc[4][4] = {};
            int kk[4], jj[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              kk[u] = min(tk * 4 + u, in - 1);
              jj[u] = min(tj + u * tjn, out - 1);
            }
            for (int p = 0; p < SP; p += 4) {
              float4 hv[4], dv[4];
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                hv[u] = *reinterpret_cast<const float4 *>(Hin + kk[u] * SP + p);
                dv[u] = *reinterpret_cast<const float4 *>(DL + jj[u] * SP + p);
              }
#pragma unroll
              for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                  acc[i][u] = fmaf(hv[i].x, dv[u].x, acc[i][u]);
                  acc[i][u] = fmaf(hv[i].y, dv[u].y, acc[i][u]);
                  acc[i][u] = fmaf(hv[i].z, dv[u].z, acc[i][u]);
                  acc[i][u] = fmaf(hv[i].w, dv[u].w, acc[i][u]);
                }
            }
            if (((in | out) & 3) == 0) {  // whole tiles: no predicates, one base address
              float *dp = dW + tk * 4 * out + tj;
#pragma unroll
              for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int u = 0; u < 4; ++u) dp[i * out + u * tjn] = acc[i][u];
            } else {
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const int k = tk * 4 + i;
                if (k >= in) continue;
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                  const int j = tj + u * tjn;
                  if (j < out) dW[k * out + j] = acc[i][u];
                }
              }
            }
          }
          float *dB = sm + P.dwp + d.b_off[l];
          for (int j = tid; j < out; j += NT) {
            float g = 0.f;
            for (int p = 0; p < SP; ++p) g += DL[j * SP + p];
            dB[j] = g;
          }
        }
        __syncthreads();
        cur ^= 1;
      }

      cluster_arrive();
      cluster_wait();  // every CTA's partial gradient is complete

      // ---- reduce slice `rank` over the cluster (4 parameters per thread), Adam in place ----
      float reg = 0.f;
      for (int i4 = 4 * tid; i4 < P.chunk; i4 += 4 * NT) {
        float4 g4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int c = 0; c < FIT_CLUSTER; ++c) {
          const float4 t = dsmem_ld4(peer[c] + (uint32_t)(P.dwp + i0 + i4) * 4u);
          g4.x += t.x; g4.y += t.y; g4.z += t.z; g4.w += t.w;
        }
        float gs[4] = {g4.x, g4.y, g4.z, g4.w};
        float outv[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int i = i0 + i4 + e;
          outv[e] = 0.f;
          if (i < i1) {
            const int off_w = tab[i] & 0xffff;
            float wv = sm[off_w], g = gs[e];
            if (a.any_l2) {
              int off_w2, off_wt2;
              float l2;
              locate(i, off_w2, off_wt2, l2);
              if (l2 != 0.f) { reg += l2 * wv * wv; g += 2.f * l2 * wv; }
            }
            float m = sm[P.am + i4 + e], v = sm[P.av + i4 + e];
            wv = opt_update<OPT>(a.opt, os, wv, g, m, v);
            sm[P.am + i4 + e] = m;
            sm[P.av + i4 + e] = v;
            outv[e] = wv;
          }
        }
        // published to the peers after the next barrier; rewritten only after the barrier that
        // follows their next backward pass, i.e. after they have all pulled it
        *reinterpret_cast<float4 *>(sm + P.wn + i4) = make_float4(outv[0], outv[1], outv[2], outv[3]);
      }
      if (a.any_l2) {
        reg = block_sum(reg, red);
        if (tid == 0) sm[P.slots + 2 + par] = reg;
      }

      cluster_arrive();
      // the next minibatch does not depend on the weights: gather it while the barrier completes
      {
        int nst = st + 1, nep = ep;
        if (nst == steps_per_epoch) { nst = 0; ++nep; }
        if (nep < epochs) gather(nep, nst);
      }
      cluster_wait();  // updated slices (and this step's loss / reg slots) are published

      // ---- pull every slice from its owner, rewrite the local W / W^T / bias images ----
      for (int i4 = 4 * tid; i4 < FIT_CLUSTER * P.chunk; i4 += 4 * NT) {
        const int c = fdiv(i4, inv_chunk), r = i4 - c * P.chunk;
        const float4 t = dsmem_ld4(peer[c] + (uint32_t)(P.wn + r) * 4u);
        const int4 cd = *reinterpret_cast<const int4 *>(tab + i4);
        const float vs[4] = {t.x, t.y, t.z, t.w};
        const int cs[4] = {cd.x, cd.y, cd.z, cd.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int off_w = cs[e] & 0xffff, off_wt = (cs[e] >> 16) - 1;
          if (off_w != 0xffff) {
            sm[off_w] = vs[e];
            if (off_wt >= 0) sm[off_wt] = vs[e];
          }
        }
      }
      if (rank == 0 && tid == 0) {
        float ls = 0.f, rg = 0.f;
        for (int c = 0; c < FIT_CLUSTER; ++c) {
          ls += dsmem_ld(peer[c] + (uint32_t)(P.slots + par) * 4u);
          if (a.any_l2) rg += dsmem_ld(peer[c] + (uint32_t)(P.slots + 2 + par) * 4u);
        }
        epoch_tot += (ls * inv_nb + rg) * (float)nb;
      }
      __syncthreads();  // images rewritten before the next forward
    }
    if (rank == 0 && tid == 0 && a.loss_out)
      a.loss_out[pb.loss0 + ep] = epoch_tot / (float)N;
  }

  // ---- write back: rank 0 the weights, every CTA its Adam slice ----
  if (rank == 0) {
    for (int l = 0; l < L; ++l) {
      const int in = d.dims[l], out = d.dims[l + 1], JP = ldo(out);
      for (int e = tid; e < in * out; e += NT) {
        const int k = e / out, j = e - k * out;
        gp[d.w_off[l] + e] = sm[P.w[l] + k * JP + j];
      }
      for (int e = tid; e < out; e += NT) gp[d.b_off[l] + e] = sm[P.b[l] + e];
    }
    if (tid == 0) run.store(a.adam_t + model, a.opt_cache + model);
  }
  for (int i = i0 + tid; i < i1; i += NT) {
    gm[i] = sm[P.am + i - i0];
    gv[i] = sm[P.av + i - i0];
  }
  cluster_arrive();
  cluster_wait();  // nobody exits while a peer may still read its shared memory
}

// the build of a kernel for an optimizer kind: OPT for every kind but Adam
template <bool W, bool R, bool E>
static auto fit_onecta_for(bool opt) { return opt ? fit_kernel<W, R, E, true> : fit_kernel<W, R, E, false>; }
template <bool W, bool E>
static auto fit_cluster_for(bool opt) { return opt ? fit_cluster_kernel<W, E, true> : fit_cluster_kernel<W, E, false>; }

// ---------------------------------------------------------------- evaluate (loss, accuracy)
__global__ void __launch_bounds__(256)
evaluate_kernel(const MlpDesc d, const float *__restrict__ params, const float *__restrict__ logits,
                const float *__restrict__ z, int N, const float *__restrict__ l2vec, const FitWeights fw,
                float *out2) {
  // logits: final pre-activation computed by K0 on a copy of the model with a linear head
  __shared__ float red[32];
  float ls = 0.f, acc = 0.f, reg = 0.f, wsum = 0.f;
  const int act_last = d.act[d.n_layers - 1];
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    const float u = logits[i], zz = z[i];
    float l = fmaxf(u, 0.f) - u * zz + log1pf(expf(-fabsf(u)));
    const float outv = act_last == BORE_ACT_SIGMOID ? stable_sigmoid(u) : u;
    float hit = ((outv > 0.5f ? 1.f : 0.f) == zz) ? 1.f : 0.f;  // Keras quirk: thresholds the OUTPUT
    if (fw.on) {
      const float ws = fit_sample_weight(fw, fw.w, i, zz);
      l *= ws; hit *= ws; wsum += ws;
    }
    ls += l;
    acc += hit;
  }
  if (l2vec)  // l2vec[2l] = kernel factor, l2vec[2l+1] = bias factor of layer l
    for (int l = 0; l < d.n_layers; ++l) {
      const int nk = d.dims[l] * d.dims[l + 1], nbias = d.dims[l + 1];
      for (int i = threadIdx.x; i < nk; i += blockDim.x) { const float w = params[d.w_off[l] + i]; reg += l2vec[2 * l] * w * w; }
      for (int i = threadIdx.x; i < nbias; i += blockDim.x) { const float w = params[d.b_off[l] + i]; reg += l2vec[2 * l + 1] * w * w; }
    }
  ls = block_sum(ls, red);
  acc = block_sum(acc, red);
  reg = block_sum(reg, red);
  if (fw.on) wsum = block_sum(wsum, red);
  if (threadIdx.x == 0) {
    out2[0] = ls / (float)N + reg;
    // weighted accuracy: Keras' Mean metric, sum(w hit) / sum(w), 0 when sum(w) = 0 (div_no_nan)
    out2[1] = fw.on ? (wsum != 0.f ? acc / wsum : 0.f) : acc / (float)N;
  }
}

constexpr size_t FIT_MAX_SMEM = 227 * 1024;

// the sample-split cluster kernel's plan; false when it does not fit (shared memory, or weight images
// too large for the 16-bit offsets of its index table)
bool fitc_plan(const MlpDesc &d, int batch, FitCPlan &p, size_t &smem) {
  make_fitc_plan(d, batch, p);
  smem = (size_t)p.total * sizeof(float);
  return smem <= 226 * 1024 && p.wend < 0xffff;
}

// the one-CTA kernel's plan for CTAs of `threads` threads; returns its shared memory in bytes
size_t fit_onecta_plan(const MlpDesc &d, int batch, int threads, int narrow, FitPlan &p) {
  make_fit_plan(d, batch, threads, 226 * 1024 / (int)sizeof(float), p, narrow);
  return (size_t)p.total * sizeof(float);
}

}  // namespace

// bore_mlp_create: automatic-mode training at batch 64 must have a kernel for one model and for many.
// Many models run the one-CTA kernel (256 threads, 128 from 2 x SMs models on); it is also where one
// model ends up when neither cluster kernel takes the net, so its plan decides both.
int fit_check_envelope(const MlpDesc &d) {
  const int B = 64;
  for (int threads : {FIT_THREADS, 128}) {
    FitPlan p;
    const size_t need = fit_onecta_plan(d, B, threads, 1, p);
    BORE_CHECK(need <= FIT_MAX_SMEM,
               "bore_mlp_create: training at batch %d needs %zu B of shared memory per model (limit %zu B)", B,
               need, FIT_MAX_SMEM);
  }
  return 0;
}

// bore_mlp_fit, bore_mlp_fit_weighted and bore_mlp_fit_ragged: the same checks and the same choice of kernel;
// fw.on == 0 runs every kernel with its unweighted arithmetic.  probs_host (ragged fits; NULL otherwise): the
// `count` problems of the launch in launch order, N the largest N_p and epochs the largest epochs_p.
static int fit_run(bore_mlp *h, int model0, int count, const float *X_dev, const float *z_dev, int N,
                   int shared_data, int batch_size, int epochs, const int32_t *perm_dev, int shared_perm,
                   float *loss_out_dev, const FitWeights &fw, void *stream,
                   const FitProblem *probs_host = nullptr) {
  BORE_CHECK(h != nullptr, "NULL handle");
  BORE_CHECK(model0 >= 0 && count >= 1 && model0 + count <= h->n_models,
             "bore_mlp_fit: models [%d,%d) outside [0,%d)", model0, model0 + count, h->n_models);
  BORE_CHECK(N >= 1 && batch_size >= 1 && epochs >= 0, "bore_mlp_fit: N=%d batch=%d epochs=%d", N,
             batch_size, epochs);
  BORE_CHECK(X_dev && z_dev && perm_dev, "bore_mlp_fit: NULL buffer");
  const int last = h->desc.act[h->desc.n_layers - 1];
  BORE_CHECK(last == BORE_ACT_SIGMOID || last == BORE_ACT_LINEAR,
             "bore_mlp_fit: binary cross-entropy needs a sigmoid or linear (from_logits) output layer");
  BORE_CUDA(cudaSetDevice(h->device));
  if (epochs == 0) return 0;
  FitArgs a;
  a.d = h->desc;
  const int B = batch_size < N ? batch_size : N;
  a.params = h->params; a.adam_m = h->adam_m; a.adam_v = h->adam_v; a.adam_t = h->adam_t;
  a.model0 = model0;
  a.X = X_dev; a.z = z_dev; a.N = N; a.shared_data = shared_data; a.batch = batch_size;
  a.epochs = epochs; a.perm = perm_dev; a.shared_perm = shared_perm;
  a.any_l2 = 0;
  for (int l = 0; l < BORE_MAX_LAYERS; ++l) {
    a.l2k[l] = l < a.d.n_layers ? h->l2k[l] : 0.f;
    a.l2b[l] = l < a.d.n_layers ? h->l2b[l] : 0.f;
    if (a.l2k[l] != 0.f || a.l2b[l] != 0.f) a.any_l2 = 1;
  }
  a.loss_out = loss_out_dev;
  a.opt = h->opt; a.opt_cache = h->opt_cache;
  a.fw = fw;
  // ragged fits: uploaded by the launch path that takes the net, after its refusals; freed on the stream after
  // the launch
  FitTable table{h, probs_host, count, (cudaStream_t)stream, {}};
  a.probs = nullptr;
  const bool ext = acts_ext(a.d.act, a.d.n_layers), opt = h->opt.kind != BORE_OPT_ADAM;
  // Tensor-pipe kernel (fit_mma.cu: 3xTF32 mma.sync GEMMs, one CTA per model) on request only (fit mode 3 or
  // BORE_FIT_MMA=1): measured SLOWER than both FFMA mappings below on B200 -- the legacy HMMA path gives
  // 3xTF32 only 1.3x the FFMA peak and every HMMA needs ~14 more instructions for fragments and splits
  // (cfg 3: 31.6 vs 20.3 ms; 4,096 cfg-4 models: 224 vs 136 ms; DESIGN.md K1t, profiles/r02_notes.md).
  {
    static int mma_env = -1;
    if (mma_env < 0) {
      const char *e = getenv("BORE_FIT_MMA");
      mma_env = e ? atoi(e) : 0;
    }
    if (h->fit_mode == 3 || (h->fit_mode == 0 && mma_env)) {
      const int rc = launch_fit_mma(h, model0, count, X_dev, z_dev, N, shared_data, batch_size, epochs, perm_dev,
                                    shared_perm, loss_out_dev, fw, table, (cudaStream_t)stream);
      if (rc != 0) return rc < 0 ? rc : 0;
      BORE_CHECK(h->fit_mode != 3, "bore_mlp_fit: the tensor-pipe kernel does not take this net / batch size");
    }
  }
  // Few models: one thread-block cluster (8 SMs) per model -- the run is latency bound and a
  // single CTA leaves the other 147 SMs idle.  Many models: one CTA each fills the GPU already.
  // First choice: the unit-split cluster kernel (fit_unit.cu, K1u); shapes it does not take (no hidden
  // layer, batch > 64, shared memory) and BORE_FIT_UNIT=0 go to the sample-split cluster kernel below.
  {
    static int unit_env = -1;
    if (unit_env < 0) {
      const char *e = getenv("BORE_FIT_UNIT");
      unit_env = e ? atoi(e) : 1;
    }
    if (h->fit_mode == 4 || (h->fit_mode == 0 && unit_env && count * FIT_CLUSTER <= h->sm_count)) {
      const int rc = launch_fit_unit(h, model0, count, X_dev, z_dev, N, shared_data, batch_size, epochs, perm_dev,
                                     shared_perm, loss_out_dev, fw, table, (cudaStream_t)stream);
      if (rc != 0) return rc < 0 ? rc : 0;
      BORE_CHECK(h->fit_mode != 4, "bore_mlp_fit: the unit-split cluster kernel does not take this net / batch size");
    }
  }
  {
    FitCPlan CP;
    size_t csmem;
    const bool fits = fitc_plan(a.d, B, CP, csmem);
    const bool want = h->fit_mode == 2 || (h->fit_mode == 0 && count * FIT_CLUSTER <= h->sm_count);
    BORE_CHECK(!(h->fit_mode == 2 && !fits), "bore_mlp_fit: cluster mode needs %zu B of shared memory", csmem);
    if (want && fits) {
      FitCArgs c;
      BORE_CHECK_RC(table.get(&a.probs));
      c.d = a.d; c.P = CP;
      c.params = a.params; c.adam_m = a.adam_m; c.adam_v = a.adam_v; c.adam_t = a.adam_t;
      c.model0 = a.model0; c.X = a.X; c.z = a.z; c.N = a.N; c.shared_data = a.shared_data;
      c.batch = a.batch; c.epochs = a.epochs; c.perm = a.perm; c.shared_perm = a.shared_perm;
      c.probs = a.probs;
      for (int l = 0; l < BORE_MAX_LAYERS; ++l) { c.l2k[l] = a.l2k[l]; c.l2b[l] = a.l2b[l]; }
      c.any_l2 = a.any_l2; c.loss_out = a.loss_out;
      c.opt = a.opt; c.opt_cache = a.opt_cache;
      c.fw = a.fw;
      const auto kern = ext ? (a.fw.on ? fit_cluster_for<true, true>(opt) : fit_cluster_for<false, true>(opt))
                            : (a.fw.on ? fit_cluster_for<true, false>(opt) : fit_cluster_for<false, false>(opt));
      BORE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)csmem));
      kern<<<count * FIT_CLUSTER, FIT_CTHREADS, csmem, (cudaStream_t)stream>>>(c);
      BORE_CUDA(cudaGetLastError());
      return 0;
    }
  }
  // threads per CTA: with more models than CTA slots the throughput is set by how many CTAs are
  // resident -- smaller CTAs, more of them (BORE_FIT_THREADS overrides).  Measured with the first
  // version of the kernel, cfg 4 (4,096 x Dense32x2 models, ms per BO iteration of all of them):
  // 256 threads 462, 128 threads 314, 64 threads 332, 32 threads 397
  int threads = count >= 2 * h->sm_count ? 128 : FIT_THREADS;
  {
    static int forced = -1;
    if (forced < 0) {
      const char *e = getenv("BORE_FIT_THREADS");
      forced = e ? atoi(e) : 0;
    }
    if (forced == 32 || forced == 64 || forced == 128 || forced == 256) threads = forced;
  }
  size_t smem;
  {
    static int narrow = -1;
    if (narrow < 0) {
      const char *e = getenv("BORE_FIT_NARROW");
      narrow = e ? atoi(e) : 1;
    }
    smem = fit_onecta_plan(a.d, B, threads, narrow, a.P);
  }
  BORE_CHECK(smem <= FIT_MAX_SMEM, "bore_mlp_fit: model + batch of %d need %zu B of shared memory", B, smem);
  BORE_CHECK_RC(table.get(&a.probs));
  const auto kern = ext ? (a.probs ? (a.fw.on ? fit_onecta_for<true, true, true>(opt) : fit_onecta_for<false, true, true>(opt))
                                   : (a.fw.on ? fit_onecta_for<true, false, true>(opt) : fit_onecta_for<false, false, true>(opt)))
                        : (a.probs ? (a.fw.on ? fit_onecta_for<true, true, false>(opt) : fit_onecta_for<false, true, false>(opt))
                                   : (a.fw.on ? fit_onecta_for<true, false, false>(opt) : fit_onecta_for<false, false, false>(opt)));
  BORE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<count, threads, smem, (cudaStream_t)stream>>>(a);
  BORE_CUDA(cudaGetLastError());
  return 0;
}

int FitTable::get(const FitProblem **out) {
  *out = static_cast<const FitProblem *>(dev.dev);
  if (!host || dev.dev) return 0;
  const size_t bytes = (size_t)n * sizeof(FitProblem);
  if (!h->tab_done) BORE_CUDA(cudaEventCreateWithFlags(&h->tab_done, cudaEventDisableTiming));
  BORE_CUDA(cudaEventSynchronize(h->tab_done));  // the previous table has left the staging buffer
  if (h->tab_cap < bytes) {
    if (h->tab_pinned) cudaFreeHost(h->tab_pinned);
    h->tab_pinned = nullptr;
    h->tab_cap = 0;
    size_t cap = 4096;
    while (cap < bytes) cap *= 2;
    BORE_CUDA(cudaMallocHost(&h->tab_pinned, cap));
    h->tab_cap = cap;
  }
  memcpy(h->tab_pinned, host, bytes);
  BORE_CUDA(dev.upload(h->tab_pinned, bytes, stream));
  BORE_CUDA(cudaEventRecord(h->tab_done, stream));
  *out = static_cast<const FitProblem *>(dev.dev);
  return 0;
}

// sample weights w (may be NULL) and class weights (cw0, cw1) -> the kernels' FitWeights; all ones is unweighted
static FitWeights fit_weights(const float *w, float cw0, float cw1) {
  FitWeights fw;
  fw.w = w; fw.cw0 = cw0; fw.cw1 = cw1;
  fw.on = w != nullptr || cw0 != 1.f || cw1 != 1.f;
  return fw;
}

static int evaluate_run(bore_mlp *h, int model, const float *X_dev, const float *z_dev, int N,
                        const FitWeights &fw, float *out_host, void *stream_) {
  BORE_CHECK(h != nullptr, "NULL handle");
  BORE_CHECK(model >= 0 && model < h->n_models, "model index %d outside [0,%d)", model, h->n_models);
  BORE_CHECK(N >= 1 && X_dev && z_dev && out_host, "bore_mlp_evaluate: bad arguments");
  BORE_CUDA(cudaSetDevice(h->device));
  cudaStream_t stream = (cudaStream_t)stream_;
  float *logits = nullptr, *out2 = nullptr;
  BORE_CUDA(cudaMalloc(&logits, (size_t)N * sizeof(float)));
  BORE_CUDA(cudaMalloc(&out2, (2 + 2 * BORE_MAX_LAYERS) * sizeof(float)));
  float l2host[2 * BORE_MAX_LAYERS];
  bool any = false;
  for (int l = 0; l < BORE_MAX_LAYERS; ++l) {
    l2host[2 * l] = l < h->desc.n_layers ? h->l2k[l] : 0.f;
    l2host[2 * l + 1] = l < h->desc.n_layers ? h->l2b[l] : 0.f;
    any = any || l2host[2 * l] != 0.f || l2host[2 * l + 1] != 0.f;
  }
  float *l2dev = out2 + 2;
  cudaMemcpyAsync(l2dev, l2host, sizeof(l2host), cudaMemcpyHostToDevice, stream);
  // forward with a linear head = the logits the loss is defined on
  bore_mlp tmp = *h;
  tmp.desc.act[tmp.desc.n_layers - 1] = BORE_ACT_LINEAR;
  int rc = launch_mlp_eval(&tmp, model, false, BORE_TRANSFORM_IDENTITY, 0, X_dev, N, logits, nullptr,
                           nullptr, nullptr, stream);
  if (!rc) {
    evaluate_kernel<<<1, 256, 0, stream>>>(h->desc, h->params + (size_t)model * h->desc.n_params,
                                           logits, z_dev, N, any ? l2dev : nullptr, fw, out2);
    cudaMemcpyAsync(out_host, out2, 2 * sizeof(float), cudaMemcpyDeviceToHost, stream);
    cudaError_t e = cudaStreamSynchronize(stream);
    if (e != cudaSuccess) { bore_set_error("bore_mlp_evaluate: %s", cudaGetErrorString(e)); rc = -2; }
  }
  cudaFree(logits);
  cudaFree(out2);
  return rc;
}

extern "C" {

int bore_mlp_fit(bore_mlp *h, int model0, int count, const float *X_dev, const float *z_dev, int N,
                 int shared_data, int batch_size, int epochs, const int32_t *perm_dev,
                 int shared_perm, float *loss_out_dev, void *stream) {
  BORE_NVTX("bore:fit (K1)");
  return fit_run(h, model0, count, X_dev, z_dev, N, shared_data, batch_size, epochs, perm_dev, shared_perm,
                 loss_out_dev, fit_weights(nullptr, 1.f, 1.f), stream);
}

int bore_mlp_fit_weighted(bore_mlp *h, int model0, int count, const float *X_dev, const float *z_dev,
                          const float *w_dev, int N, int shared_data, float class_weight0,
                          float class_weight1, int batch_size, int epochs, const int32_t *perm_dev,
                          int shared_perm, float *loss_out_dev, void *stream) {
  BORE_NVTX("bore:fit weighted (K1)");
  return fit_run(h, model0, count, X_dev, z_dev, N, shared_data, batch_size, epochs, perm_dev, shared_perm,
                 loss_out_dev, fit_weights(w_dev, class_weight0, class_weight1), stream);
}

int bore_mlp_fit_ragged(bore_mlp *h, int model0, int count, const float *X_dev, const float *z_dev,
                        const float *w_dev, const int32_t *n_host, const int32_t *epochs_host, float class_weight0,
                        float class_weight1, int batch_size, const int32_t *perm_dev, float *loss_out_dev,
                        void *stream) {
  BORE_NVTX("bore:fit ragged (K1)");
  BORE_CHECK(h != nullptr, "NULL handle");
  BORE_CHECK(model0 >= 0 && count >= 1 && count <= h->n_models - model0,
             "bore_mlp_fit_ragged: models [%d,%d) outside [0,%d)", model0, model0 + count, h->n_models);
  BORE_CHECK(n_host && epochs_host, "bore_mlp_fit_ragged: NULL count array");
  BORE_CHECK(X_dev && z_dev && perm_dev, "bore_mlp_fit_ragged: NULL buffer");
  BORE_CHECK(batch_size >= 1, "bore_mlp_fit_ragged: batch=%d", batch_size);
  const long long D = h->desc.dims[0];
  // every problem gets its descriptor; the ones with epochs_p = 0 are not launched (their state is untouched)
  std::vector<FitProblem> probs;
  std::vector<long long> work;
  long long R = 0, Q = 0, E = 0;
  int maxN = 0, maxE = 0;
  for (int p = 0; p < count; ++p) {
    const int n = n_host[p], e = epochs_host[p];
    BORE_CHECK(n >= 1 && e >= 0, "bore_mlp_fit_ragged: problem %d has N=%d, epochs=%d", p, n, e);
    FitProblem f;
    f.row0 = R; f.perm0 = Q; f.loss0 = E;
    f.model = model0 + p; f.N = n; f.epochs = e; f.pad_ = 0;
    long long rows_x, ne;
    BORE_CHECK(!__builtin_add_overflow(R, (long long)n, &R) && !__builtin_mul_overflow(R, D, &rows_x) &&
                   !__builtin_mul_overflow((long long)n, (long long)e, &ne) &&
                   !__builtin_add_overflow(Q, ne, &Q) && !__builtin_add_overflow(E, (long long)e, &E),
               "bore_mlp_fit_ragged: the sizes overflow 64 bits at problem %d", p);
    if (e == 0) continue;
    probs.push_back(f);
    work.push_back((long long)e * (((long long)n + batch_size - 1) / batch_size));
    maxN = n > maxN ? n : maxN;
    maxE = e > maxE ? e : maxE;
  }
  // launch order: longest problem first (Adam steps), ties in problem order, so that a long problem does not
  // start in the last wave of CTAs (DESIGN.md, "Ragged batched problems").  BORE_FIT_RAGGED_ORDER=0 launches
  // in problem order (read on every call: lets one process time both orders).  Results do not depend on it.
  const char *order_env = getenv("BORE_FIT_RAGGED_ORDER");
  if (!(order_env && order_env[0] == '0')) {
    std::vector<int> idx(probs.size());
    for (size_t i = 0; i < idx.size(); ++i) idx[i] = (int)i;
    std::stable_sort(idx.begin(), idx.end(), [&](int x, int y) { return work[x] > work[y]; });
    std::vector<FitProblem> sorted(probs.size());
    for (size_t i = 0; i < idx.size(); ++i) sorted[i] = probs[idx[i]];
    probs.swap(sorted);
  }
  return fit_run(h, model0, probs.empty() ? count : (int)probs.size(), X_dev, z_dev, probs.empty() ? 1 : maxN,
                 0, batch_size, maxE, perm_dev, 0, loss_out_dev, fit_weights(w_dev, class_weight0, class_weight1),
                 stream, probs.empty() ? nullptr : probs.data());
}

int bore_mlp_set_fit_mode(bore_mlp *h, int mode) {
  BORE_CHECK(h != nullptr, "NULL handle");
  BORE_CHECK(mode >= 0 && mode <= 4, "bore_mlp_set_fit_mode: mode %d outside [0,4]", mode);
  h->fit_mode = mode;
  return 0;
}

int bore_mlp_evaluate(bore_mlp *h, int model, const float *X_dev, const float *z_dev, int N,
                      float *out_host, void *stream) {
  return evaluate_run(h, model, X_dev, z_dev, N, fit_weights(nullptr, 1.f, 1.f), out_host, stream);
}

int bore_mlp_evaluate_weighted(bore_mlp *h, int model, const float *X_dev, const float *z_dev,
                               const float *w_dev, float class_weight0, float class_weight1, int N,
                               float *out_host, void *stream) {
  return evaluate_run(h, model, X_dev, z_dev, N, fit_weights(w_dev, class_weight0, class_weight1), out_host,
                      stream);
}

}  // extern "C"
