// K1t: fused classifier training on the TENSOR pipe (sm_100a) -- the whole Keras `fit` of one model in
// one CTA, every GEMM of a minibatch step as 3xTF32 `mma.sync.m16n8k8` (error-compensated split:
// a = a_hi + a_lo, a b ~ a_lo b_hi + a_hi b_lo + a_hi b_hi, fp32 accumulation -- fp32-level accuracy).
//
// Replaces keras Model.fit (README.rst:66,93; bore/plugins/hpbandster/base.py:156-157,184), like
// fit.cu's two FFMA kernels, which remain the path for shapes this kernel does not take.
//
// Why tensor cores here (north_star: "only if ncu shows tensor-pipe utilisation beats the FP32 FFMA
// path"): a single model is 10^3 strictly dependent steps of 4 MFLOP.  On FFMA that is 16k issue cycles
// per step for ONE SM (8.2 us at 100 % efficiency), which is why fit.cu spreads a model over an 8-CTA
// cluster and then pays two cluster barriers, a DSMEM gradient reduction and a 46 KB weight pull per
// step (20.7 us per step measured).  On the tensor pipe the nine GEMMs of a step are ~100 mma per warp
// each, one SM is enough, nothing leaves the CTA, and the step is bounded by ~9 CTA barriers.
//
// Layout.  Activations [sample][unit] and weights [in][out] row-major in shared memory, every leading
// dimension == 8 (mod 32): the four fragment access patterns a step needs (A and A', B and B') are then
// all bank-conflict free with plain LDS, so ONE weight image serves forward, reverse and update:
//   forward   H_l     = act(H_{l-1} W_l + b_l)               A = H_{l-1} [b][k],  B = W_l [k][n]
//   reverse   D_{l-1} = (D_l W_l') . act'(H_{l-1})           A = D_l [b][j],      B(k=j, n=i) = W_l[i][j]
//   update    dW_l    = H_{l-1}' D_l                         A(m=i, k=b) = H_{l-1}[b][i],  B = D_l [b][n]
// Weights are kept PRE-SPLIT as (hi, lo) float2 pairs, hi = w rounded to TF32, lo = w - hi (exact), so the
// pair IS the fp32 master value and the B operand of forward and reverse is one LDS.64 with no conversion
// (each weight is read by 8 warps per step but written once); leading dimension == 4 (mod 16) pairs.
// Activations and deltas are split on the fly (3 instructions per element: integer round-to-TF32, subtract;
// the tensor core ignores the low 13 bits of lo).  The first version used cvt.rna.tf32.f32 -- ~10 SASS
// instructions each on sm_100a -- and predicated mma inside runtime-sized tile groups: 28.8 executed
// instructions per HMMA, 38.4 ms per cfg-3 fit (profiles/r02_notes.md); every tile-group size is now a
// template instance.
// The thread that holds a dW accumulator owns that weight: Keras-form Adam straight from the fragment
// (slots m, v stream through L2, requested before the GEMM that produces the gradient).  The next
// minibatch is gathered by cp.async while the reverse pass runs.
#include <stdlib.h>

#include "common.cuh"
#include "fit_common.cuh"

namespace {

constexpr int MT_MAXB = 64;  // minibatch rows (4 m16 blocks)
constexpr int MT_TPW = 4;    // weight-gradient tiles one warp may own per layer (kernel template: 1, 2 or 4)

struct FitMPlan {
  int L;                          // Dense layers incl. the 1-unit output layer
  int kp[BORE_MAX_LAYERS];        // in  padded to 8  (K of forward, N of reverse)
  int np[BORE_MAX_LAYERS];        // out padded to 8  (N of forward / update, K of reverse)
  int mp[BORE_MAX_LAYERS];        // in  padded to 16 (M of update)
  int ldw[BORE_MAX_LAYERS];
  int w[BORE_MAX_LAYERS];         // weight image [kp][ldw] (output layer: vector [kp])
  int b[BORE_MAX_LAYERS];         // bias [np]
  int bm[BORE_MAX_LAYERS], bv[BORE_MAX_LAYERS];  // Adam slots of the biases (whole run in smem)
  int wm, wv;                     // Adam slots of the output layer's kernel [kp]
  int tpw[BORE_MAX_LAYERS];       // update tiles per warp
  int ngf[BORE_MAX_LAYERS];       // n-tiles per warp unit in the forward GEMM of layer l (1, 2 or 4)
  int ngb[BORE_MAX_LAYERS];       // ... in the reverse GEMM of layer l (output width = np[l-1])
  int ldx, lda;
  int x[2], zb[2], idx[2];        // minibatch double buffer: rows [64][ldx], labels, row indices
  int h[BORE_MAX_LAYERS];         // hidden activations [64][lda]
  int s;                          // spare [64][lda]: delta ping-pong partner
  int du;                         // dL/dlogit [64]
  int cs[2];                      // column-sum partials of the deltas [4][lda] (bias gradients)
  int red;                        // [32]
  int total;
};

inline int ld_for(int v) { return v + ((8 - v % 32) + 32) % 32; }  // smallest >= v that is 8 mod 32
inline int ldp_for(int v) { return v + ((4 - v % 16) + 16) % 16; } // smallest >= v that is 4 mod 16 (float2 units)
// n-tiles per warp unit: the widest group (4, 2, 1) that divides the row of tiles and still leaves a unit per warp
inline int pick_ng(int mblocks, int ntn, int nwarps) {
  for (int ng = 4; ng > 1; ng >>= 1)
    if (ntn % ng == 0 && mblocks * (ntn / ng) >= nwarps) return ng;
  return 1;
}
inline int r4i(int v) { return (v + 3) & ~3; }

// false: this net / batch is not taken by the tensor kernel (the caller falls back to fit.cu)
bool make_fitm_plan(const MlpDesc &d, int B, int nwarps, FitMPlan &p) {
  const int L = d.n_layers;
  if (L < 2 || L > BORE_MAX_LAYERS || d.dims[L] != 1 || B > MT_MAXB) return false;
  p.L = L;
  int off = 0, maxnp = 8;
  for (int l = 0; l < L; ++l) {
    const int in = d.dims[l], out = d.dims[l + 1];
    p.kp[l] = round_up(in, 8);
    p.np[l] = round_up(out, 8);
    p.mp[l] = round_up(in, 16);
    if (l < L - 1) {
      if (p.np[l] > 128) return false;
      if (p.np[l] > maxnp) maxnp = p.np[l];
      p.ldw[l] = ldp_for(p.np[l]);
      p.ngf[l] = pick_ng((B + 15) / 16, p.np[l] / 8, nwarps);
      p.ngb[l] = l > 0 ? pick_ng((B + 15) / 16, p.np[l - 1] / 8, nwarps) : 1;
      const int ntn = p.np[l] / 8, tiles = (p.mp[l] / 16) * ntn;
      int tpw = (tiles + nwarps - 1) / nwarps;
      while (tpw <= MT_TPW && (ntn % tpw || tpw == 3)) ++tpw;
      if (tpw > MT_TPW) return false;
      p.tpw[l] = tpw;
      p.w[l] = off; off += r4i(2 * p.kp[l] * p.ldw[l]);
    } else {
      p.ldw[l] = 1; p.tpw[l] = 0; p.ngf[l] = p.ngb[l] = 1;
      p.w[l] = off; off += r4i(p.kp[l]);
      p.wm = off; off += r4i(p.kp[l]);
      p.wv = off; off += r4i(p.kp[l]);
    }
    p.b[l] = off; off += r4i(p.np[l]);
    p.bm[l] = off; off += r4i(p.np[l]);
    p.bv[l] = off; off += r4i(p.np[l]);
  }
  p.ldx = ld_for(p.mp[0]);
  p.lda = ld_for(maxnp + 8);  // (+8: the update GEMM reads columns up to mp = in padded to 16)
  for (int i = 0; i < 2; ++i) {
    p.x[i] = off; off += MT_MAXB * p.ldx;
    p.zb[i] = off; off += MT_MAXB;
    p.idx[i] = off; off += MT_MAXB;
  }
  for (int l = 0; l < L - 1; ++l) { p.h[l] = off; off += MT_MAXB * p.lda; }
  p.s = off; off += MT_MAXB * p.lda;
  p.du = off; off += MT_MAXB;
  p.cs[0] = off; off += 4 * p.lda;
  p.cs[1] = off; off += 4 * p.lda;
  p.red = off; off += 32;
  p.total = r4i(off);
  return true;
}

struct FitMArgs {
  MlpDesc d;
  FitMPlan P;
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

// ------------------------------------------------------------------------------------ mma plumbing
// a = hi + lo with hi = a rounded to TF32 (integer round-half-up on the magnitude) and lo = a - hi, which is
// exact; the tensor core reads the top 19 bits of lo.  3 instructions.
__device__ __forceinline__ void split_tf32(float a, uint32_t &hi, uint32_t &lo) {
  hi = (__float_as_uint(a) + 0x1000u) & 0xffffe000u;
  lo = __float_as_uint(a - __uint_as_float(hi));
}
__device__ __forceinline__ float2 split_pair(float a) {
  uint32_t hi, lo;
  split_tf32(a, hi, lo);
  return make_float2(__uint_as_float(hi), __uint_as_float(lo));
}
__device__ __forceinline__ void mma_tf32(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// the three products of the compensated scheme, small terms first
__device__ __forceinline__ void mma_3x(float (&c)[4], const uint32_t (&ah)[4], const uint32_t (&al)[4], uint32_t bh0,
                                       uint32_t bl0, uint32_t bh1, uint32_t bl1) {
  mma_tf32(c, al, bh0, bh1);
  mma_tf32(c, ah, bl0, bl1);
  mma_tf32(c, ah, bh0, bh1);
}

// Fragment layout of m16n8k8 (g = lane / 4, t = lane % 4): a0 (g, t) a1 (g+8, t) a2 (g, t+4) a3 (g+8, t+4);
// b0 (k = t, n = g) b1 (k = t+4, n = g); c0 (g, 2t) c1 (g, 2t+1), c2 c3 the same columns of row g+8.
//
// A operand from a raw fp32 matrix, A(m, k) = A[m a_rs + k a_cs], split on the fly.
struct AFrag {
  uint32_t h[4], l[4];
};
__device__ __forceinline__ void load_a(AFrag &f, const float *pa, int a8, int a4) {
  split_tf32(pa[0], f.h[0], f.l[0]);
  split_tf32(pa[a8], f.h[1], f.l[1]);
  split_tf32(pa[a4], f.h[2], f.l[2]);
  split_tf32(pa[a8 + a4], f.h[3], f.l[3]);
}

// acc[q] += A[m0.., :K] W[:K, n0 + 8q..] -- B from a pre-split weight image, B(k, n) = Wp[k b_rs + n b_cs] (pairs)
template <int NG>
__device__ __forceinline__ void gemm_w(const float *__restrict__ A, int a_rs, const float2 *__restrict__ Wp, int b_rs,
                                       int b_cs, int m0, int n0, int K, float (&acc)[NG][4], int lane) {
  const int g = lane >> 2, t = lane & 3;
  const float *pa = A + (m0 + g) * a_rs + t;
  const float2 *pb = Wp + t * b_rs + (n0 + g) * b_cs;
  const int a8 = 8 * a_rs, b4 = 4 * b_rs, b8 = 8 * b_cs, bk = 8 * b_rs;
#pragma unroll 2
  for (int k0 = 0; k0 < K; k0 += 8) {
    AFrag f;
    load_a(f, pa, a8, 4);
#pragma unroll
    for (int q = 0; q < NG; ++q) {
      const float2 w0 = pb[q * b8], w1 = pb[q * b8 + b4];
      mma_3x(acc[q], f.h, f.l, __float_as_uint(w0.x), __float_as_uint(w0.y), __float_as_uint(w1.x),
             __float_as_uint(w1.y));
    }
    pa += 8;
    pb += bk;
  }
}

// acc[q] += H[:K, m0..]' D[:K, n0 + 8q..] -- the weight-gradient GEMM: both operands raw, K = minibatch rows
template <int NG>
__device__ __forceinline__ void gemm_hd(const float *__restrict__ H, int h_rs, const float *__restrict__ Dl, int d_rs,
                                        int m0, int n0, int K, float (&acc)[NG][4], int lane) {
  const int g = lane >> 2, t = lane & 3;
  const float *pa = H + t * h_rs + m0 + g;   // A(m = i, k = b) = H[b][i]
  const float *pb = Dl + t * d_rs + n0 + g;  // B(k = b, n = j) = D[b][j]
  const int a4 = 4 * h_rs, b4 = 4 * d_rs;
#pragma unroll 2
  for (int k0 = 0; k0 < K; k0 += 8) {
    AFrag f;
    load_a(f, pa, 8, a4);
#pragma unroll
    for (int q = 0; q < NG; ++q) {
      uint32_t bh0, bl0, bh1, bl1;
      split_tf32(pb[q * 8], bh0, bl0);
      split_tf32(pb[q * 8 + b4], bh1, bl1);
      mma_3x(acc[q], f.h, f.l, bh0, bl0, bh1, bl1);
    }
    pa += 8 * h_rs;
    pb += 8 * d_rs;
  }
}

__device__ __forceinline__ void cp_async4(float *dst_smem, const float *src) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst_smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// forward unit: NG tiles of H_l = act(A W_l + b_l), rows mb*16.., columns n0..
template <int NG, bool EXT>
__device__ __forceinline__ void fwd_unit(const float *A, int a_rs, const float2 *Wp, int ldw, const float *bs, float *H,
                                         int lda, int mb, int n0, int K, int act, int lane) {
  const int g = lane >> 2, t = lane & 3;
  float acc[NG][4];
#pragma unroll
  for (int q = 0; q < NG; ++q) acc[q][0] = acc[q][1] = acc[q][2] = acc[q][3] = 0.f;
  gemm_w<NG>(A, a_rs, Wp, ldw, 1, mb * 16, n0, K, acc, lane);
#pragma unroll
  for (int q = 0; q < NG; ++q) {
    const int n = n0 + q * 8 + 2 * t;
    const float2 b = *reinterpret_cast<const float2 *>(bs + n);
    float *h0 = H + (mb * 16 + g) * lda + n;
    *reinterpret_cast<float2 *>(h0) = make_float2(act_fwd<EXT>(act, acc[q][0] + b.x), act_fwd<EXT>(act, acc[q][1] + b.y));
    *reinterpret_cast<float2 *>(h0 + 8 * lda) = make_float2(act_fwd<EXT>(act, acc[q][2] + b.x), act_fwd<EXT>(act, acc[q][3] + b.y));
  }
}

// reverse unit: NG tiles of D_{l-1} = (D_l W_l') . act'(H_{l-1}) and their column sums (bias gradient partials)
template <int NG, bool EXT>
__device__ __forceinline__ void bwd_unit(const float *Dl, int lda, const float2 *Wp, int ldw, const float *Hin, int h_rs,
                                         float *DN, float *cs, int mb, bool live, int n0, int K, int actp, int lane) {
  const int g = lane >> 2, t = lane & 3;
  float acc[NG][4];
#pragma unroll
  for (int q = 0; q < NG; ++q) acc[q][0] = acc[q][1] = acc[q][2] = acc[q][3] = 0.f;
  if (live) gemm_w<NG>(Dl, lda, Wp, 1, ldw, mb * 16, n0, K, acc, lane);  // B(k = j, n = i) = W[i][j]
#pragma unroll
  for (int q = 0; q < NG; ++q) {
    const int n = n0 + q * 8 + 2 * t;
    float2 d0 = make_float2(0.f, 0.f), d1 = d0;
    if (live) {
      const float *h0 = Hin + (mb * 16 + g) * h_rs + n;
      const float2 hv0 = *reinterpret_cast<const float2 *>(h0);
      const float2 hv1 = *reinterpret_cast<const float2 *>(h0 + 8 * h_rs);
      d0 = make_float2(acc[q][0] * act_bwd<EXT>(actp, hv0.x), acc[q][1] * act_bwd<EXT>(actp, hv0.y));
      d1 = make_float2(acc[q][2] * act_bwd<EXT>(actp, hv1.x), acc[q][3] * act_bwd<EXT>(actp, hv1.y));
      float *o0 = DN + (mb * 16 + g) * lda + n;
      *reinterpret_cast<float2 *>(o0) = d0;
      *reinterpret_cast<float2 *>(o0 + 8 * lda) = d1;
    }
    float s0 = d0.x + d1.x, s1 = d0.y + d1.y;  // rows g and g + 8; then over g by shuffle
#pragma unroll
    for (int o = 4; o < 32; o <<= 1) {
      s0 += __shfl_xor_sync(0xffffffffu, s0, o);
      s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    }
    if (g == 0) *reinterpret_cast<float2 *>(cs + mb * lda + n) = make_float2(s0, s1);
  }
}

// ------------------------------------------------------------------------------------ the kernel
template <int NW, int TPW, bool EXT, bool OPT>
__global__ void __launch_bounds__(NW * 32, NW >= 16 ? 1 : (NW >= 8 ? 2 : 4)) fit_mma_kernel(const FitMArgs a) {
  extern __shared__ __align__(16) float sm[];
  const MlpDesc &d = a.d;
  const FitMPlan &P = a.P;
  constexpr int NT = NW * 32;
  const int L = P.L, LH = P.L - 1;  // LH hidden layers; layer LH is the 1-unit output layer
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const FitProblem pb = fit_problem(a, blockIdx.x);
  const int model = pb.model, N = pb.N, epochs = pb.epochs;
  float *gp = a.params + (size_t)model * d.n_params;
  float *gm = a.adam_m + (size_t)model * d.n_params;
  float *gv = a.adam_v + (size_t)model * d.n_params;
  const float *X = a.X + pb.row0 * d.dims[0];
  const float *zg = a.z + pb.row0;
  const int *perm = a.perm + pb.perm0;
  const float *wg = a.fw.w ? a.fw.w + pb.row0 : nullptr;
  const int D = d.dims[0], lda = P.lda, ldx = P.ldx;
  float *red = sm + P.red;

  // ---- stage: zero everything (padding must be finite zeros), then weights, biases, Adam slots ----
  for (int e = tid; e < P.total; e += NT) sm[e] = 0.f;
  __syncthreads();
  for (int l = 0; l < L; ++l) {
    const int in = d.dims[l], out = d.dims[l + 1];
    if (l < LH) {
      const int ldw = P.ldw[l];
      float2 *Wp = reinterpret_cast<float2 *>(sm + P.w[l]);
      for (int e = tid; e < in * out; e += NT) {
        const int k = e / out, j = e - k * out;
        Wp[k * ldw + j] = split_pair(gp[d.w_off[l] + e]);
      }
    } else {
      for (int e = tid; e < in; e += NT) {
        sm[P.w[l] + e] = gp[d.w_off[l] + e];
        sm[P.wm + e] = gm[d.w_off[l] + e];
        sm[P.wv + e] = gv[d.w_off[l] + e];
      }
    }
    for (int e = tid; e < out; e += NT) {
      sm[P.b[l] + e] = gp[d.b_off[l] + e];
      sm[P.bm[l] + e] = gm[d.b_off[l] + e];
      sm[P.bv[l] + e] = gv[d.b_off[l] + e];
    }
  }
  OptRun<OPT> run(a.opt, a.adam_t[model], a.opt_cache + model);
  OptStep os = OptRun<OPT>::consts(a.opt);
  const int spe = (N + a.batch - 1) / a.batch;
  const int total_steps = epochs * spe;

  // row index of sample `tid` of global step `gs` (threads < 64; -1 beyond the batch): requested a step
  // ahead so that its latency hides behind the forward pass; rows and labels follow by cp.async
  auto row_of = [&](int gs) {
    int row = -1;
    if (tid < MT_MAXB && gs < total_steps) {
      const int ep = gs / spe, st = gs - ep * spe;
      const int s0 = st * a.batch, nb = min(a.batch, N - s0);
      if (tid < nb) row = __ldg(perm + (size_t)ep * N + s0 + tid);
    }
    return row;
  };
  const float inv_D = 1.f / (float)D;
  auto issue_rows = [&](int buf) {
    const int *idx = reinterpret_cast<const int *>(sm + P.idx[buf]);
    float *xb = sm + P.x[buf];
    for (int e = tid; e < MT_MAXB * D; e += NT) {
      const int p = fdiv(e, inv_D), k = e - p * D;
      const int row = idx[p];
      if (row >= 0) cp_async4(xb + p * ldx + k, X + (size_t)row * D + k);
      else xb[p * ldx + k] = 0.f;
    }
    if (tid < MT_MAXB) {
      const int row = idx[tid];
      if (row >= 0) cp_async4(sm + P.zb[buf] + tid, zg + row);
      else sm[P.zb[buf] + tid] = 0.f;
      // sample weights into dL/dlogit's slot: dead from the end of the output-layer phase (this is issued
      // after it) to the next loss, which reads a sample's weight before it writes its dL/dlogit there
      if (wg) {
        if (row >= 0) cp_async4(sm + P.du + tid, wg + row);
        else sm[P.du + tid] = 0.f;
      }
    }
    cp_async_commit();
  };
  __syncthreads();
  if (tid < MT_MAXB) reinterpret_cast<int *>(sm + P.idx[0])[tid] = row_of(0);
  __syncthreads();
  if (total_steps > 0) issue_rows(0);

  // Adam on the update tiles this warp owns of layer `l` (gradients in acc, slots in mm / vv)
  float reg = 0.f;
  auto adam_tiles = [&](int l, float (&acc)[TPW][4], float (&mm)[TPW][4], float (&vv)[TPW][4]) {
    const int in = d.dims[l], out = d.dims[l + 1], ldw = P.ldw[l], ntn = P.np[l] >> 3, tpw = P.tpw[l];
    const int T0 = warp * tpw;
    if (T0 >= (P.mp[l] >> 4) * ntn) return;
    const int mb = T0 / ntn, nt0 = T0 - mb * ntn;
    float2 *Wp = reinterpret_cast<float2 *>(sm + P.w[l]);
    const float l2 = a.l2k[l];
#pragma unroll
    for (int q = 0; q < TPW; ++q) {
      if (q < tpw) {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int i = mb * 16 + g + (c >> 1) * 8, j = (nt0 + q) * 8 + 2 * t + (c & 1);
          if (i < in && j < out) {
            const float2 wp = Wp[i * ldw + j];
            float wv = wp.x + wp.y;  // the fp32 master value, exactly
            float gr = acc[q][c];
            if (l2 != 0.f) { reg += l2 * wv * wv; gr += 2.f * l2 * wv; }
            float m = mm[q][c], v = vv[q][c];
            wv = opt_update<OPT>(a.opt, os, wv, gr, m, v);
            const int gi = d.w_off[l] + i * out + j;
            gm[gi] = m; gv[gi] = v;
            Wp[i * ldw + j] = split_pair(wv);
          }
        }
      }
    }
  };

  float epoch_tot = 0.f;
  for (int gs = 0; gs < total_steps; ++gs) {
    const int cur = gs & 1;
    const int ep = gs / spe, st = gs - ep * spe;
    const int nb = min(a.batch, N - st * a.batch);
    const int nmb = (nb + 15) >> 4, BP = nmb << 4;
    const float inv_nb = 1.f / (float)nb;
    reg = 0.f;
    run.advance(a.opt, os);

    const int row_next = row_of(gs + 1);  // (consumed after the forward pass)
    cp_async_wait_all();
    __syncthreads();  // the minibatch is in; every weight update of the previous step is visible

    // ---- forward through the hidden layers ----
    for (int l = 0; l < LH; ++l) {
      const float *A = l == 0 ? sm + P.x[cur] : sm + P.h[l - 1];
      const int a_rs = l == 0 ? ldx : lda;
      const float2 *Wp = reinterpret_cast<const float2 *>(sm + P.w[l]);
      const float *bs = sm + P.b[l];
      float *H = sm + P.h[l];
      const int ldw = P.ldw[l], ntn = P.np[l] >> 3, act = d.act[l], K = P.kp[l], ng = P.ngf[l];
      const int groups = ntn / ng;
      for (int u = warp; u < nmb * groups; u += NW) {
        const int mb = u / groups, n0 = (u - mb * groups) * ng * 8;
        if (ng == 4) fwd_unit<4, EXT>(A, a_rs, Wp, ldw, bs, H, lda, mb, n0, K, act, lane);
        else if (ng == 2) fwd_unit<2, EXT>(A, a_rs, Wp, ldw, bs, H, lda, mb, n0, K, act, lane);
        else fwd_unit<1, EXT>(A, a_rs, Wp, ldw, bs, H, lda, mb, n0, K, act, lane);
      }
      __syncthreads();
    }

    // ---- output layer: logit, loss, dL/dlogit (mean over the batch); a warp per row ----
    {
      const float *H = sm + P.h[LH - 1];
      const float *w = sm + P.w[LH];
      const float b = sm[P.b[LH]];
      const int in = P.kp[LH];
      float lsum = 0.f;
      for (int r = warp; r < BP; r += NW) {
        const float wr = wg ? sm[P.du + r] : 1.f;  // (read before the shuffles, written after them)
        float u = 0.f;
        for (int k = lane; k < in; k += 32) u = fmaf(H[r * lda + k], w[k], u);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) u += __shfl_xor_sync(0xffffffffu, u, o);
        u += b;
        float dl = 0.f;
        if (r < nb) {
          const float zz = sm[P.zb[cur] + r];
          float l = fmaxf(u, 0.f) - u * zz + log1pf(expf(-fabsf(u))), g = stable_sigmoid(u) - zz;
          if (a.fw.on) {
            const float ws = wr * (zz != 0.f ? a.fw.cw1 : a.fw.cw0);
            l *= ws; g *= ws;
          }
          lsum += l;
          dl = g * inv_nb;
        }
        if (lane == 0) sm[P.du + r] = dl;
      }
      if (lane == 0) red[warp] = lsum;
    }
    if (tid < MT_MAXB) reinterpret_cast<int *>(sm + P.idx[cur ^ 1])[tid] = row_next;  // (free since the last step)
    __syncthreads();

    // ---- delta of the top hidden layer (into the spare buffer), output-layer gradients + Adam ----
    float wl_new = 0.f, bl_new = 0.f;  // the output layer's new parameters, written after the barrier
    {
      const float *H = sm + P.h[LH - 1];
      const float *du = sm + P.du;
      const float *w = sm + P.w[LH];
      float *DN = sm + P.s;
      float *cs = sm + P.cs[0];
      const int npv = P.np[LH - 1], actp = d.act[LH - 1];
      // thread = one column j and every RG-th row (RG row groups)
      const int RG = NT / npv > 0 ? min(NT / npv, 4) : 1;
      if (tid < npv * RG) {
        const int j = tid % npv, rg = tid / npv;
        const float wj = w[j];
        float csum = 0.f;
        for (int r = rg; r < BP; r += RG) {
          const float hv = H[r * lda + j];
          const float dv = du[r] * wj * act_bwd<EXT>(actp, hv);
          DN[r * lda + j] = dv;
          csum += dv;
        }
        cs[rg * lda + j] = csum;
        for (int r2 = RG; r2 < 4; ++r2) if (rg == 0) cs[r2 * lda + j] = 0.f;
      }
      // dw[k] = sum_b H[b][k] du[b] by the LAST warps (the first ones carry the loop above)
      const int in = d.dims[LH];
      const int tb = NT - 1 - tid;
      if (tb < in) {
        float gk = 0.f;
        for (int r = 0; r < BP; ++r) gk = fmaf(H[r * lda + tb], du[r], gk);
        float wv = w[tb];
        const float l2 = a.l2k[LH];
        if (l2 != 0.f) { reg += l2 * wv * wv; gk += 2.f * l2 * wv; }
        float m = sm[P.wm + tb], v = sm[P.wv + tb];
        wl_new = opt_update<OPT>(a.opt, os, wv, gk, m, v);
        sm[P.wm + tb] = m; sm[P.wv + tb] = v;
      } else if (tb == in) {
        float gb = 0.f;
        for (int r = 0; r < BP; ++r) gb += du[r];
        float bv = sm[P.b[LH]];
        const float l2 = a.l2b[LH];
        if (l2 != 0.f) { reg += l2 * bv * bv; gb += 2.f * l2 * bv; }
        float m = sm[P.bm[LH]], v = sm[P.bv[LH]];
        bl_new = opt_update<OPT>(a.opt, os, bv, gb, m, v);
        sm[P.bm[LH]] = m; sm[P.bv[LH]] = v;
      }
      if (tid == 0) {  // the step's data loss (fixed order)
        float ls = 0.f;
        for (int w2 = 0; w2 < NW; ++w2) ls += red[w2];
        epoch_tot += ls * inv_nb * (float)nb;
      }
    }
    __syncthreads();
    {
      const int in = d.dims[LH];
      const int tb = NT - 1 - tid;
      if (tb < in) sm[P.w[LH] + tb] = wl_new;
      else if (tb == in) sm[P.b[LH]] = bl_new;
    }
    if (gs + 1 < total_steps) issue_rows(cur ^ 1);  // next minibatch: lands while the reverse pass runs

    // ---- reverse through the hidden layers: D_{l-1}, dW_l, Adam ----
    // delta_l sits in `dbuf`; delta_{l-1} goes to the buffer of H_l (dead once delta_l exists) / the spare
    const float *dbuf = sm + P.s;
    int csi = 0;                       // cs[csi] holds the column sums of delta_l
    float accp[TPW][4];                // dW of the layer above, waiting for its Adam pass
    float mp_[TPW][4], vp_[TPW][4];
    int lp = -1;                       // that layer (-1: none pending)
    for (int l = LH - 1; l >= 0; --l) {
      const int in = d.dims[l], out = d.dims[l + 1], ldw = P.ldw[l], ntn = P.np[l] >> 3, tpw = P.tpw[l];
      const float *Hin = l == 0 ? sm + P.x[cur] : sm + P.h[l - 1];
      const int h_rs = l == 0 ? ldx : lda;
      // (0) Adam of the layer above (its reverse GEMM was completed before the last barrier)
      if (lp >= 0) adam_tiles(lp, accp, mp_, vp_);
      // (1) bias of this layer from the column sums of delta_l
      if (tid < out) {
        const float *cs = sm + P.cs[csi];
        float gb = (cs[tid] + cs[lda + tid]) + (cs[2 * lda + tid] + cs[3 * lda + tid]);
        float bv = sm[P.b[l] + tid];
        const float l2 = a.l2b[l];
        if (l2 != 0.f) { reg += l2 * bv * bv; gb += 2.f * l2 * bv; }
        float m = sm[P.bm[l] + tid], v = sm[P.bv[l] + tid];
        bv = opt_update<OPT>(a.opt, os, bv, gb, m, v);
        sm[P.bm[l] + tid] = m; sm[P.bv[l] + tid] = v;
        sm[P.b[l] + tid] = bv;
      }
      // (2) request the Adam slots of the tiles this warp will own
      float mm[TPW][4], vv[TPW][4];
      const int T0 = warp * tpw;
      const bool own = T0 < (P.mp[l] >> 4) * ntn;
      const int mbw = own ? T0 / ntn : 0, nt0 = own ? T0 - mbw * ntn : 0;
#pragma unroll
      for (int q = 0; q < TPW; ++q)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          mm[q][c] = 0.f; vv[q][c] = 0.f;
          if (own && q < tpw) {
            const int i = mbw * 16 + g + (c >> 1) * 8, j = (nt0 + q) * 8 + 2 * t + (c & 1);
            if (i < in && j < out) {
              const int gi = d.w_off[l] + i * out + j;
              mm[q][c] = __ldcg(gm + gi); vv[q][c] = __ldcg(gv + gi);
            }
          }
        }
      // (3) delta_{l-1} = (delta_l W_l') . act'(H_{l-1}) and its column sums
      if (l > 0) {
        float *DN = (dbuf == sm + P.s) ? sm + P.h[l] : sm + P.s;
        const float2 *Wp = reinterpret_cast<const float2 *>(sm + P.w[l]);
        const int nti = P.np[l - 1] >> 3, actp = d.act[l - 1], K = P.np[l], ng = P.ngb[l];
        float *cs = sm + P.cs[csi ^ 1];
        const int groups = nti / ng;
        for (int u = warp; u < 4 * groups; u += NW) {  // all four row blocks: dead ones publish zero column sums
          const int mb = u / groups, n0 = (u - mb * groups) * ng * 8;
          const bool live = mb < nmb;
          if (ng == 4) bwd_unit<4, EXT>(dbuf, lda, Wp, ldw, Hin, h_rs, DN, cs, mb, live, n0, K, actp, lane);
          else if (ng == 2) bwd_unit<2, EXT>(dbuf, lda, Wp, ldw, Hin, h_rs, DN, cs, mb, live, n0, K, actp, lane);
          else bwd_unit<1, EXT>(dbuf, lda, Wp, ldw, Hin, h_rs, DN, cs, mb, live, n0, K, actp, lane);
        }
      }
      // (4) dW_l = H_{l-1}' delta_l on the tiles this warp owns
      float acc[TPW][4];
#pragma unroll
      for (int q = 0; q < TPW; ++q) acc[q][0] = acc[q][1] = acc[q][2] = acc[q][3] = 0.f;
      if (own) {
        if (TPW == 1 || tpw == TPW) {
          gemm_hd<TPW>(Hin, h_rs, dbuf, lda, mbw * 16, nt0 * 8, BP, acc, lane);
        } else if (TPW == 4 && tpw == 2) {
          float a2[2][4] = {};
          gemm_hd<2>(Hin, h_rs, dbuf, lda, mbw * 16, nt0 * 8, BP, a2, lane);
#pragma unroll
          for (int c = 0; c < 4; ++c) { acc[0][c] = a2[0][c]; acc[1][c] = a2[1][c]; }
        } else {
          float a1[1][4] = {};
          gemm_hd<1>(Hin, h_rs, dbuf, lda, mbw * 16, nt0 * 8, BP, a1, lane);
#pragma unroll
          for (int c = 0; c < 4; ++c) acc[0][c] = a1[0][c];
        }
      }
      if (l == 0) {
        adam_tiles(0, acc, mm, vv);  // nobody reads W_0 in this phase: no barrier needed before its update
      } else {
#pragma unroll
        for (int q = 0; q < TPW; ++q)
#pragma unroll
          for (int c = 0; c < 4; ++c) { accp[q][c] = acc[q][c]; mp_[q][c] = mm[q][c]; vp_[q][c] = vv[q][c]; }
        dbuf = (dbuf == sm + P.s) ? sm + P.h[l] : sm + P.s;
        csi ^= 1;
        __syncthreads();
      }
      lp = l;
    }
    if (a.any_l2) {
      const float r = block_sum(reg, red);
      if (tid == 0) epoch_tot += r * (float)nb;
    }
    if (st == spe - 1) {
      if (tid == 0 && a.loss_out) a.loss_out[pb.loss0 + ep] = epoch_tot / (float)N;
      epoch_tot = 0.f;
    }
  }

  // ---- write the trained weights and the smem-resident Adam slots back ----
  cp_async_wait_all();
  __syncthreads();
  for (int l = 0; l < L; ++l) {
    const int in = d.dims[l], out = d.dims[l + 1];
    if (l < LH) {
      const int ldw = P.ldw[l];
      const float2 *Wp = reinterpret_cast<const float2 *>(sm + P.w[l]);
      for (int e = tid; e < in * out; e += NT) {
        const int k = e / out, j = e - k * out;
        const float2 wp = Wp[k * ldw + j];
        gp[d.w_off[l] + e] = wp.x + wp.y;
      }
    } else {
      for (int e = tid; e < in; e += NT) {
        gp[d.w_off[l] + e] = sm[P.w[l] + e];
        gm[d.w_off[l] + e] = sm[P.wm + e];
        gv[d.w_off[l] + e] = sm[P.wv + e];
      }
    }
    for (int e = tid; e < out; e += NT) {
      gp[d.b_off[l] + e] = sm[P.b[l] + e];
      gm[d.b_off[l] + e] = sm[P.bm[l] + e];
      gv[d.b_off[l] + e] = sm[P.bv[l] + e];
    }
  }
  if (tid == 0) run.store(a.adam_t + model, a.opt_cache + model);
}

template <int NW, int TPW>
int launch_cfg(const FitMArgs &a, int count, size_t smem, cudaStream_t stream) {
  const bool ext = acts_ext(a.d.act, a.d.n_layers), opt = a.opt.kind != BORE_OPT_ADAM;
  const auto kern = ext ? (opt ? fit_mma_kernel<NW, TPW, true, true> : fit_mma_kernel<NW, TPW, true, false>)
                        : (opt ? fit_mma_kernel<NW, TPW, false, true> : fit_mma_kernel<NW, TPW, false, false>);
  BORE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<count, NW * 32, smem, stream>>>(a);
  BORE_CUDA(cudaGetLastError());
  return 0;
}
template <int NW>
int launch_nw(const FitMArgs &a, int count, size_t smem, cudaStream_t stream) {
  int tpw = 1;
  for (int l = 0; l < a.P.L - 1; ++l) tpw = a.P.tpw[l] > tpw ? a.P.tpw[l] : tpw;
  if (tpw == 1) return launch_cfg<NW, 1>(a, count, smem, stream);
  if (tpw == 2) return launch_cfg<NW, 2>(a, count, smem, stream);
  return launch_cfg<NW, 4>(a, count, smem, stream);
}

}  // namespace

// 1: launched; 0: shape not taken by the tensor kernel (caller falls back); < 0: error
int launch_fit_mma(const bore_mlp *h, int model0, int count, const float *X_dev, const float *z_dev, int N,
                   int shared_data, int batch_size, int epochs, const int32_t *perm_dev, int shared_perm,
                   float *loss_out_dev, const FitWeights &fw, FitTable &tab, cudaStream_t stream) {
  const int B = batch_size < N ? batch_size : N;
  // few models: one 16-warp CTA per model (latency); many: 4-warp CTAs, several per SM (throughput)
  int nw = count * 2 <= h->sm_count ? 16 : (count <= 2 * h->sm_count ? 8 : 4);
  {
    static int forced = -1;
    if (forced < 0) {
      const char *e = getenv("BORE_FIT_MMA_WARPS");
      forced = e ? atoi(e) : 0;
    }
    if (forced == 4 || forced == 8 || forced == 16) nw = forced;
  }
  FitMArgs a;
  a.d = h->desc;
  bool ok = false;
  for (; nw <= 16; nw *= 2) {  // a wide layer may need more warps to own its update tiles
    if (make_fitm_plan(a.d, B, nw, a.P)) { ok = true; break; }
  }
  if (!ok) return 0;
  const size_t smem = (size_t)a.P.total * sizeof(float);
  if (smem > 227 * 1024) return 0;
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
  {
    const int rc = tab.get(&a.probs);  // taken: the table goes up now
    if (rc) return rc;
  }
  int rc;
  if (nw == 16) rc = launch_nw<16>(a, count, smem, stream);
  else if (nw == 8) rc = launch_nw<8>(a, count, smem, stream);
  else rc = launch_nw<4>(a, count, smem, stream);
  return rc < 0 ? rc : 1;
}
