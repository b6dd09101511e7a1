// K1u: fused classifier training, ONE model = one thread-block cluster, hidden UNITS split over the CTAs.
//
// Same job as fit.cu (the whole Keras Model.fit with Adam + binary cross-entropy in one launch;
// README.rst:66,93, bore/plugins/hpbandster/base.py:156-157,184), other decomposition.  The first
// cluster kernel (fit_cluster_kernel) splits the SAMPLES of a minibatch over 8 CTAs: every CTA holds
// all weights, carries 8 samples through the net, and each step ends with a reduce-scatter of 8
// partial gradients, Adam on a parameter slice and an all-gather of the new weights into two weight
// images -- 54,600 warp instructions per CTA and step, 22 barriers, 20.5 us per step on B200
// (profiles/r02c_notes.md).  Here CTA r of the cluster OWNS units [r U, (r+1) U) of every
// hidden layer:
//   * forward, layer l: h_{l+1}[:, slice] = act(h_l Wc_l + b) from the column slice Wc_l = W_l[:, slice]
//     over ALL samples of the minibatch; the slice (U rows, contiguous) goes into every peer's copy of
//     h_{l+1} by ONE bulk copy per peer (cp.async.bulk shared::cta -> shared::cluster) that completes its
//     bytes on the PEER's mbarrier; a CTA waits until the seven other slices have landed in its own copy
//     and for nothing else (no barrier.cluster, no per-thread remote stores);
//   * the Dense(1) output layer, the loss, dL/dlogit and the delta of the last hidden layer are
//     computed by every CTA for itself (a few thousand flops: cheaper than one exchange);
//   * reverse, layer l: delta_l[:, slice] = (delta_{l+1} Wr_l') . act'(h_l[:, slice]) from the row slice
//     Wr_l = W_l[slice, :], pushed like the activations (the delta of the first hidden layer stays local);
//   * weight gradients: a CTA computes dW only for the two slices it stores (Wc_l and Wr_l) from the
//     complete activations / deltas it holds; Adam follows in place for all of them with every thread.
//     No gradient reduction, no weight exchange, no second weight image: the only traffic between SMs
//     is the activations (4 x 7 x 2.2 KB out of every CTA per step at cfg 3).
// W_l[k][j] is therefore updated twice, by the owner of column j (in Wc_l) and by the owner of row k
// (in Wr_l).  Both run the same instructions on the same operands in the same order (the sample sum
// is a packed FFMA2 chain over even / odd samples of each half of the minibatch, halves and lanes added
// in a fixed order), so the two copies stay bit-identical for the whole run; the column copies are what
// is written back.
//
// GEMM mapping inside a CTA (512 threads, out = U units x SP samples, K <= 64..): the K dimension is
// split over FU_KS = 4 WARPS (16 consecutive k each), a lane holds an 8-sample x 2-unit register tile
// (eight LDS.128 of activations + two of weights per four k, 32 FFMA2), the partial tiles meet in a shared
// scratch [warp][unit][sample] and 128 threads sum the partials of four outputs each in a fixed tree, apply
// bias / activation (or act') and store the slice.  One __syncthreads per half; no shuffles.  K is padded
// to a multiple of 16 with zero weights (one trip of four k per warp).  The pass is bound by shared-memory wavefronts and by the latency
// of its dependent chain, not by issue slots: all 16 warps splitting K cost more (16 partial copies: 32 KB
// written and read back per pass), 8 warps the same as 4.
//
// Rows of every activation / delta buffer are SP + 4 floats apart: the gradient tiles read 8 different
// rows per quarter warp with LDS.128, which this stride spreads over all 32 banks.  Weights are unit-major
// (one row per own unit, the reduction index along the row): the Adam pass walks them linearly.
//
// A CTA cannot run more than one exchange ahead of the slowest peer (it needs everybody's slice to go on),
// which is what makes single buffers safe for everything but h_1 (pushed first in a step, while peers may
// still read last step's h_1 for their weight gradients -- two buffers, alternating).
//
// History (profiles/r02c_notes.md): plain remote stores + barrier.cluster 15.4 ms per cfg-3 fit (10 % of the
// time in MEMBAR, 13 % at the barrier); st.async + mbarrier 14.5; compile-time shapes 12.8; bulk-copy
// exchange, unit-major weights, 4 x 4 gradient tiles over two sample halves, Adam as its own pass 11.3.
// The sample-split cluster kernel (fit.cu, fit mode 2): 20.4.
//
// The kernel is compiled for run-time shapes and, because a step is ~35,000 mostly scalar instructions of
// index arithmetic around short FFMA2 bursts, again with the shape as template constants for the uniform
// nets of BASELINE.json (hidden width 16 / 32 / 64, batch 64): strides, trip counts and layer loops fold
// (cfg 3: 15.4 ms run-time shapes, 11.3 ms compile-time).
#include <stdlib.h>

//#define FU_TRACE 1
#include "common.cuh"
#include "fit_common.cuh"

namespace {

constexpr int FU_C = 8;          // CTAs per cluster (portable maximum)
constexpr int FU_THREADS = 512;
constexpr int FU_NW = FU_THREADS / 32;  // warps
constexpr int FU_KT = 16;          // K is padded to a multiple of this: 4 consecutive k per trip for each of the FU_KS warps
constexpr int FU_NBAR = 3 * BORE_MAX_LAYERS + 2;

__host__ __device__ constexpr int fu_r2(int a) { return (a + 1) & ~1; }
__host__ __device__ constexpr int fu_r4(int a) { return (a + 3) & ~3; }
__host__ __device__ constexpr int fu_r8(int a) { return (a + 7) & ~7; }
__host__ __device__ constexpr int fu_rk(int a) { return (a + FU_KT - 1) / FU_KT * FU_KT; }
__host__ __device__ constexpr int fu_max(int a, int b) { return a > b ? a : b; }
__host__ __device__ constexpr int fu_kps(int a) { return fu_rk(a) + 4; }

struct FuPlan {
  int SP, SPP;                      // padded batch (multiple of 8) and row stride SP + 4
  int U[BORE_MAX_LAYERS + 1];       // U[i], i = 1..L-1: units of hidden layer i per CTA (even)
  // one copy of this CTA's parameters (floats); Adam m / v and the gradient follow at + npar / + 2 npar /
  // + 3 npar.  Matrices are UNIT-major: one row per own unit, kps(n) = rk(n) + 4 floats long (the reduction
  // index runs along the row: consecutive lanes update consecutive addresses; + 4 keeps the rows of the four
  // unit pairs of a warp in different banks), zero beyond the layer's width (never updated)
  int wc[BORE_MAX_LAYERS];          // l = 0..L-2: Wc_l  [U[l+1]][kps(dims[l])]
  int wr[BORE_MAX_LAYERS];          // l = 1..L-2: Wr_l  [U[l]][kps(dims[l+1])]   (row slice)
  int bs[BORE_MAX_LAYERS];          // l = 0..L-2: bias slice [U[l+1]]
  int wl, bl;                       // output layer [dims[L-1]], [1] (every CTA holds and updates it)
  int npar;
  int par0;                         // offset of the parameter block
  int h0[2];                        // minibatch [rk(dims[0])][SPP], double buffered (prefetch)
  int h[BORE_MAX_LAYERS][2];        // h_i, i = 1..L-1: [max(C U[i], rk(dims[i]))][SPP]; second buffer for i == 1
  int dg[BORE_MAX_LAYERS];          // delta_i complete, i = 2..L-1 (i == L-1: computed locally), rows as h_i
  int d1;                           // delta_1: this CTA's slice [U[1]][SPP] when L > 2, else = dg[1] complete
  int scratch, wstride;             // [FU_KS][wstride = umax * SP]
  int lg;                           // logit partials [FU_THREADS / SP][SP]
  int dz, zb, idx;                  // dL/dlogit [SP]; labels [2][SP]; row indices of the next step [SP] (ints)
  int wb;                           // sample weights of a weighted fit [SP]
  int slots;                        // lsum[2][2], reg[2]
  int bars;                         // mbarriers (8 bytes each): h_i at 2 (i - 1) + buffer, delta_i at 2 L + i
  int total;
};

__host__ __device__ inline bool make_fu_plan(const MlpDesc &d, int batch, FuPlan &p) {
  const int L = d.n_layers;
  if (L < 2 || d.dims[L] != 1) return false;
  p.SP = fu_r8(batch);
  p.SPP = p.SP + 4;
  if (p.SP > FU_THREADS) return false;
  int off = 0, umax = 0;
  for (int i = 1; i <= L - 1; ++i) {
    p.U[i] = fu_r2((d.dims[i] + FU_C - 1) / FU_C);
    if (p.U[i] > umax) umax = p.U[i];
  }
  int np = 0;
  for (int l = 0; l <= L - 2; ++l) { p.wc[l] = np; np += fu_kps(d.dims[l]) * p.U[l + 1]; }
  for (int l = 1; l <= L - 2; ++l) { p.wr[l] = np; np += fu_kps(d.dims[l + 1]) * p.U[l]; }
  for (int l = 0; l <= L - 2; ++l) { p.bs[l] = np; np += p.U[l + 1]; }
  p.wl = np; np += d.dims[L - 1];
  p.bl = np; np += 1;
  p.npar = fu_r4(np);
  p.par0 = off; off += 5 * p.npar;  // w | m | v | gradient, first half of the samples | second half
  p.h0[0] = off; off += fu_rk(d.dims[0]) * p.SPP;
  p.h0[1] = off; off += fu_rk(d.dims[0]) * p.SPP;
  for (int i = 1; i <= L - 1; ++i) {
    const int rows = fu_max(FU_C * p.U[i], fu_rk(d.dims[i]));
    p.h[i][0] = off; off += rows * p.SPP;
    p.h[i][1] = p.h[i][0];
    if (i == 1) { p.h[i][1] = off; off += rows * p.SPP; }
  }
  for (int i = 2; i <= L - 1; ++i) { p.dg[i] = off; off += fu_max(FU_C * p.U[i], fu_rk(d.dims[i])) * p.SPP; }
  if (L > 2) { p.d1 = off; off += p.U[1] * p.SPP; }
  else { p.dg[1] = off; p.d1 = off; off += fu_max(FU_C * p.U[1], fu_rk(d.dims[1])) * p.SPP; }
  p.wstride = umax * p.SP;
  p.scratch = off; off += fu_max(4, 32 / 4) * p.wstride;  // FU_KS partial copies (+ room for block_sum)
  p.lg = off; off += (FU_THREADS / p.SP) * p.SP;
  p.dz = off; off += p.SP;
  p.zb = off; off += 2 * p.SP;
  p.idx = off; off += p.SP;
  // one buffer: the loss reads it before the barrier after which the next step's weights are requested
  p.wb = off; off += p.SP;
  p.slots = off; off += 8;
  off = fu_r2(off);  // mbarriers are 8 bytes
  p.bars = off; off += 2 * FU_NBAR;
  p.total = fu_r4(off);
  return true;
}

struct FuArgs : FitJob {
  FuPlan P;
};

// ---------------------------------------------------------------- cluster / packed-FMA primitives
__device__ __forceinline__ uint32_t fu_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void fu_cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t fu_peer(const void *p, uint32_t rank) {
  uint32_t a = (uint32_t)__cvta_generic_to_shared(p), r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(rank));
  return r;
}
// one bulk copy (TMA engine) of a contiguous block of this CTA's shared memory into a peer's, completing `bytes`
// on the PEER's mbarrier -- the exchange costs the sender one instruction per peer instead of per-thread remote
// stores (which, at 4,096 x 4 B and later 1,024 x 16 B per CTA and exchange, kept the LSU / MIO port busy for
// ~1,500 cycles after every push and slowed whatever followed: clock64 trace in profiles/r02c_notes.md)
__device__ __forceinline__ void fu_bulk_push(uint32_t dst, uint32_t src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "r"(src), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void fu_fence_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fu_bar_init(uint32_t bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fu_bar_expect(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void fu_bar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "FU_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra FU_DONE;\n"
      "bra FU_WAIT;\n"
      "FU_DONE:\n"
      "}\n" ::"r"(bar),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ float fu_ld(uint32_t addr) {
  float v;
  asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
  return v;
}
// FFMA2 (PTX fma.rn.f32x2): two IEEE fp32 FMAs per instruction, the same roundings as two fmaf
typedef unsigned long long fu_u64;
__device__ __forceinline__ fu_u64 fu_pk(float lo, float hi) {
  fu_u64 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void fu_fma2(fu_u64 &c, fu_u64 a, fu_u64 b) {
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(c) : "l"(a), "l"(b));
}
__device__ __forceinline__ float2 fu_upk(fu_u64 v) {
  float2 r;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(v));
  return r;
}

// ---------------------------------------------------------------- GEMM pass, first half
// scratch[w][u * SP + s] = sum over warp w's k of A[k][s] * Wm[u][k]     (w < FU_KS, u < U, s < SP)
// A: [KP][SPP], Wm: [U][KP + 4], KP a multiple of 64 (zero beyond the layer's width in Wm).  Warp w takes
// k in [w KP / KS, (w + 1) KP / KS); lane tile: samples {4 so .. 4 so + 3} and {SP/2 + 4 so ..}, units 2 up, 2 up + 1.
// Why only FU_KS of the 16 warps: the pass is bound by shared-memory wavefronts, not by issue slots.  With
// all 16 warps splitting K the 16 partial copies of the output were 32 KB written and 32 KB read back per pass
// (~1,050 cycles per pass measured with clock64); with 4 warps x 16 k the loads are 10 LDS.128 per 32 FFMA2
// and the partials 8 KB each way.
constexpr int FU_KS = 4;
static_assert(FU_KT == 4 * FU_KS, "K is padded to one trip of four k per k-split warp");
__device__ __forceinline__ void fu_partial(const float *__restrict__ A, const float *__restrict__ Wm, int KP, int U,
                                           int SP, int SPP, float inv_nso, float *__restrict__ mine, int warp, int lane) {
  const int nso = SP >> 3, ntile = nso * (U >> 1), half = SP >> 1;
  const int kw = KP / FU_KS, kps = KP + 4;
  for (int tile = lane; tile < ntile; tile += 32) {
    const int up = fdiv(tile, inv_nso), so = tile - up * nso;
    ulonglong2 acc[2][2];  // [unit][sample quad]: .x = samples (0, 1), .y = samples (2, 3) of the quad
#pragma unroll
    for (int e = 0; e < 2; ++e)
#pragma unroll
      for (int i = 0; i < 2; ++i) acc[e][i] = make_ulonglong2(0ull, 0ull);
    const float *ap = A + 4 * so + warp * kw * SPP;
    const float *wp = Wm + 2 * up * kps + warp * kw;
    // four consecutive k per trip, all ten loads in flight before the first FFMA2
    for (int k0 = 0; k0 < kw; k0 += 4) {
      float4 a0[4], a1[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        a0[i] = *reinterpret_cast<const float4 *>(ap + i * SPP);
        a1[i] = *reinterpret_cast<const float4 *>(ap + i * SPP + half);
      }
      const float4 wa = *reinterpret_cast<const float4 *>(wp), wb = *reinterpret_cast<const float4 *>(wp + kps);
      ap += 4 * SPP;
      wp += 4;
      const float w0s[4] = {wa.x, wa.y, wa.z, wa.w}, w1s[4] = {wb.x, wb.y, wb.z, wb.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const fu_u64 a01 = fu_pk(a0[i].x, a0[i].y), a23 = fu_pk(a0[i].z, a0[i].w);
        const fu_u64 a45 = fu_pk(a1[i].x, a1[i].y), a67 = fu_pk(a1[i].z, a1[i].w);
        const fu_u64 w0 = fu_pk(w0s[i], w0s[i]), w1 = fu_pk(w1s[i], w1s[i]);
        fu_fma2(acc[0][0].x, a01, w0); fu_fma2(acc[0][0].y, a23, w0); fu_fma2(acc[0][1].x, a45, w0); fu_fma2(acc[0][1].y, a67, w0);
        fu_fma2(acc[1][0].x, a01, w1); fu_fma2(acc[1][0].y, a23, w1); fu_fma2(acc[1][1].x, a45, w1); fu_fma2(acc[1][1].y, a67, w1);
      }
    }
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      float *o = mine + (2 * up + e) * SP + 4 * so;
      *reinterpret_cast<ulonglong2 *>(o) = acc[e][0];
      *reinterpret_cast<ulonglong2 *>(o + half) = acc[e][1];
    }
  }
}

// ---------------------------------------------------------------- GEMM pass, second half
// epi(u, s4, sums of the FU_KS partials of outputs (u, s4 .. s4 + 3)) for u < U, s4 = 0, 4, .. < SP
template <class Epi>
__device__ __forceinline__ void fu_reduce(const float *__restrict__ scratch, int U, int SP, float inv_nq, int wstride,
                                          Epi epi) {
  const int nq = SP >> 2, n = U * nq;
  for (int o = threadIdx.x; o < n; o += FU_THREADS) {
    float4 p[FU_KS];
#pragma unroll
    for (int w = 0; w < FU_KS; ++w) p[w] = *reinterpret_cast<const float4 *>(scratch + w * wstride + 4 * o);
#pragma unroll
    for (int st = 1; st < FU_KS; st <<= 1)
#pragma unroll
      for (int w = 0; w < FU_KS; w += 2 * st) {
        p[w].x += p[w + st].x; p[w].y += p[w + st].y; p[w].z += p[w + st].z; p[w].w += p[w + st].w;
      }
    const int u = fdiv(o, inv_nq);
    epi(u, 4 * (o - u * nq), p[0]);
  }
}

// One 4 x 4 block of a weight gradient: g[e][i] = sum_s RB_e[s] * RA_i[s] over s < SP, as an even / odd
// packed chain (FFMA2 on (s, s + 1) pairs), lo + hi at the end.  Operand order does not matter (the
// products commute), so the column copy (A = activations, B = deltas) and the row copy (A = deltas,
// B = activations) of the same weight get the same bits.  8 LDS.128 per 32 FFMA2: the phase is bound by
// shared-memory wavefronts (every lane reads its own rows) and by the half-rate FFMA2 pipe of the few warps
// that hold tiles (4 x 2 tiles over all samples: 4,200 cycles for cfg 3), hence the sample range is cut in
// two halves that go to different warps; the halves are added in the Adam pass (fixed order).
__device__ __forceinline__ void fu_grad_tile(const float *__restrict__ const (&ar)[4], const float *__restrict__ const (&br)[4],
                                             int s_lo, int s_hi, float (&g)[4][4]) {
  fu_u64 acc[4][4];
#pragma unroll
  for (int e = 0; e < 4; ++e)
#pragma unroll
    for (int i = 0; i < 4; ++i) acc[e][i] = 0ull;
#pragma unroll 2
  for (int s = s_lo; s < s_hi; s += 4) {
    float4 x[4], y[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) x[i] = *reinterpret_cast<const float4 *>(ar[i] + s);
#pragma unroll
    for (int e = 0; e < 4; ++e) y[e] = *reinterpret_cast<const float4 *>(br[e] + s);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const fu_u64 ya = fu_pk(y[e].x, y[e].y), yb = fu_pk(y[e].z, y[e].w);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        fu_fma2(acc[e][i], fu_pk(x[i].x, x[i].y), ya);
        fu_fma2(acc[e][i], fu_pk(x[i].z, x[i].w), yb);
      }
    }
  }
#pragma unroll
  for (int e = 0; e < 4; ++e)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 v = fu_upk(acc[e][i]);
      g[e][i] = v.x + v.y;
    }
}
// the same chain for one row pair (output layer)
__device__ __forceinline__ float fu_row_dot(const float *__restrict__ a, const float *__restrict__ b, int SP) {
  fu_u64 acc = 0ull;
#pragma unroll 4
  for (int s = 0; s < SP; s += 4) {
    const float4 x = *reinterpret_cast<const float4 *>(a + s), y = *reinterpret_cast<const float4 *>(b + s);
    fu_fma2(acc, fu_pk(x.x, x.y), fu_pk(y.x, y.y));
    fu_fma2(acc, fu_pk(x.z, x.w), fu_pk(y.z, y.w));
  }
  const float2 v = fu_upk(acc);
  return v.x + v.y;
}
__device__ __forceinline__ float fu_row_sum(const float *__restrict__ a, int SP) {
  float e = 0.f, o = 0.f;
#pragma unroll 4
  for (int s = 0; s < SP; s += 4) {
    const float4 x = *reinterpret_cast<const float4 *>(a + s);
    e += x.x; o += x.y; e += x.z; o += x.w;
  }
  return e + o;
}

// NH > 0: the net has NH hidden layers of HW units each (HW a multiple of 16) and the padded batch is SPT --
// compile-time shape, D stays a run-time value; NH == 0: everything from the descriptor and the plan.
// WT: per-sample loss weights (FuArgs::fw); the unweighted build runs none of their code.
// EXT: the activation codes above BORE_ACT_TANH (act.cuh).  OPT: the optimizers other than Adam (opt.cuh).
// DROP (with OPT only): dropout after the hidden layers (dropout.cuh).
template <int NH, int HW, int SPT, bool WT, bool EXT, bool OPT, bool DROP>
__global__ void __cluster_dims__(FU_C, 1, 1) __launch_bounds__(FU_THREADS) fit_unit_kernel(const FuArgs a) {
  extern __shared__ __align__(16) float sm[];
  constexpr bool FIX = NH > 0;
  constexpr int ML = FIX ? NH : BORE_MAX_LAYERS - 1;  // bound of the unrolled loops over hidden layers
  const MlpDesc &d = a.d;
  const FuPlan &P = a.P;
  const int D = d.dims[0];
  const int L = FIX ? NH + 1 : d.n_layers;
  const int SP = FIX ? SPT : P.SP, SPP = SP + 4;
  // width of layer l's output (l = 0: the input), units per CTA of hidden layer i
#define FU_DIM(l) (FIX ? ((l) == 0 ? D : ((l) > NH ? 1 : HW)) : d.dims[l])
#define FU_U(i) (FIX ? HW / FU_C : P.U[i])
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int rank = (int)fu_rank();
  const FitProblem pb = fit_problem(a, blockIdx.x / FU_C);  // which problem of the launch
  const int model = pb.model, N = pb.N, epochs = pb.epochs;
  float *gp = a.params + (size_t)model * d.n_params;
  float *gm = a.adam_m + (size_t)model * d.n_params;
  float *gv = a.adam_v + (size_t)model * d.n_params;
  const float *X = a.X + pb.row0 * D;
  const float *zg = a.z + pb.row0;
  const int *perm = a.perm + pb.perm0;
  const float *wg = WT && a.fw.w ? a.fw.w + pb.row0 : nullptr;
  const int steps_per_epoch = (N + a.batch - 1) / a.batch;
  float *W = sm + P.par0, *Mm = W + P.npar, *Vv = Mm + P.npar, *Gg = Vv + P.npar;
  const int wstride = FIX ? (HW / FU_C) * SPT : P.wstride;  // floats per warp of the scratch
  const float inv_sp = 1.f / (float)SP, inv_nso = 1.f / (float)(SP >> 3), inv_nq = 1.f / (float)(SP >> 2);

  // ---- zero everything, then stage this CTA's parameter slices and their Adam slots ----
  for (int i = tid; i < P.total; i += FU_THREADS) sm[i] = 0.f;
  __syncthreads();
  const uint32_t bars = (uint32_t)__cvta_generic_to_shared(sm + P.bars);  // local mbarriers, 8 bytes apart
  if (tid == 0) {
    for (int i = 0; i < FU_NBAR; ++i) fu_bar_init(bars + 8u * i, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int l = 0; l <= L - 2; ++l) {
    const int in = d.dims[l], out = d.dims[l + 1], U = P.U[l + 1], kps = fu_kps(in);
    for (int e = tid; e < in * U; e += FU_THREADS) {
      const int k = e / U, u = e - k * U, j = rank * U + u;
      if (j < out) {
        const int gi = d.w_off[l] + k * out + j, pi = P.wc[l] + u * kps + k;
        W[pi] = gp[gi]; Mm[pi] = gm[gi]; Vv[pi] = gv[gi];
      }
    }
    for (int u = tid; u < U; u += FU_THREADS) {
      const int j = rank * U + u;
      if (j < out) {
        const int gi = d.b_off[l] + j;
        W[P.bs[l] + u] = gp[gi]; Mm[P.bs[l] + u] = gm[gi]; Vv[P.bs[l] + u] = gv[gi];
      }
    }
  }
  for (int l = 1; l <= L - 2; ++l) {
    const int in = d.dims[l], out = d.dims[l + 1], U = P.U[l], kps = fu_kps(out);
    for (int e = tid; e < out * U; e += FU_THREADS) {
      const int u = e / out, j = e - u * out, k = rank * U + u;
      if (k < in) {
        const int gi = d.w_off[l] + k * out + j, pi = P.wr[l] + u * kps + j;
        W[pi] = gp[gi]; Mm[pi] = gm[gi]; Vv[pi] = gv[gi];
      }
    }
  }
  for (int k = tid; k <= d.dims[L - 1]; k += FU_THREADS) {  // output layer: weights, then the bias
    const int gi = k < d.dims[L - 1] ? d.w_off[L - 1] + k : d.b_off[L - 1];
    W[P.wl + k] = gp[gi]; Mm[P.wl + k] = gm[gi]; Vv[P.wl + k] = gv[gi];
  }
  OptRun<OPT> run(a.opt, a.adam_t[model], a.opt_cache + model);
  uint32_t peer[FU_C];  // base of every CTA's dynamic shared memory
#pragma unroll
  for (int c = 0; c < FU_C; ++c) peer[c] = fu_peer(sm, c);

  // ---- minibatch prefetch: cp.async (4 bytes each) straight into h0[next][k][p], transposing by address ----
  // step top         warps that idle during the GEMM passes read the row indices of the NEXT step -> idx (shared)
  // gradient phase   every warp takes whole rows (sample p = warp, warp + 16, ...; lane = feature k, k + 32, ...:
  //                  coalesced global reads) and copies them element by element; awaited before the barrier that
  //                  ends the step.  Padded samples: zero fill (src-size 0).
  // Whichever way the 12.8 KB of a cfg-3 minibatch are requested, the step pays ~1,500 cycles for them (clock64
  // traces, profiles/r02c_notes.md).  Tried: loads into registers + a commit pass, lanes along p (32 rows per
  // request) or along k, by all threads or by the warps that idle in the GEMM passes (fence.proxy.async of the
  // next exchange then waits for them); cp.async into a staging tile + transposition in the Adam pass; one bulk
  // copy (TMA) per row -- cp.async.bulk issues lane after lane through the uniform datapath, ~55 cycles each, and
  // keeps its warp from the next barrier; the same dealt over idle warps and windows; cp.async by the three
  // warps without a work item (32 shared-memory rows per request: ~80 cycles per instruction, 8,000 in all).
  // This form, spread over all warps, was the cheapest together with the register form: 23,100 - 23,900 cycles per
  // step against 25,000 - 27,800 for the others.
  int *idxs = reinterpret_cast<int *>(sm + P.idx);
  auto row_of = [&](int ep, int st, int p) -> int {
    const int s0 = st * a.batch;
    const int nb = min(a.batch, N - s0);
    return p < nb ? perm[(size_t)ep * N + s0 + p] : -1;
  };
  const int gt = tid - 32 * FU_KS;  // thread index among the warps that idle during the GEMM passes
  auto index_stage = [&](int ep, int st) {  // visible after the next __syncthreads
    if (gt >= 0 && gt < SP) idxs[gt] = row_of(ep, st, gt);
  };
  auto cp4 = [&](float *dst, const float *src, bool valid) {
    const uint32_t d32 = (uint32_t)__cvta_generic_to_shared(dst);
    const int n = valid ? 4 : 0;
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(d32), "l"(src), "r"(n) : "memory");
  };
  auto gather_async = [&](int buf, int w0) {  // warps w0 .. FU_NW - 1
    if (warp < w0) return;
    float *H0 = sm + P.h0[buf];
    for (int p = warp - w0; p < SP; p += FU_NW - w0) {
      const int row = idxs[p];
      const float *xr = X + (size_t)max(row, 0) * D;
      for (int k = lane; k < D; k += 32) cp4(H0 + k * SPP + p, xr + k, row >= 0);
      if (lane == 0) {
        cp4(sm + P.zb + buf * SP + p, zg + max(row, 0), row >= 0);
        if (wg) cp4(sm + P.wb + p, wg + max(row, 0), row >= 0);
      }
    }
  };
  auto gather_wait = [&]() { asm volatile("cp.async.wait_all;" ::: "memory"); };
  index_stage(0, 0);
  __syncthreads();
  gather_async(0, 0);
  gather_wait();
  fu_cluster_sync();  // everybody's shared memory and mbarriers exist and are initialised

  const int NLG = FU_THREADS / SP;  // k-parts of the logit
  const int HL = FU_DIM(L - 1);
  int n_tiles = 0, n_items = 0;
#pragma unroll
  for (int l = 0; l < ML; ++l)
    if (l <= L - 2) n_tiles += ((FU_DIM(l) + 3) >> 2) * ((FU_U(l + 1) + 3) >> 2);
#pragma unroll
  for (int l = 1; l < ML; ++l)
    if (l <= L - 2) n_tiles += ((FU_DIM(l + 1) + 3) >> 2) * ((FU_U(l) + 3) >> 2);
  n_items = 2 * n_tiles + HL + 1;  // every tile twice: first / second half of the samples
#pragma unroll
  for (int l = 0; l < ML; ++l)
    if (l <= L - 2) n_items += FU_U(l + 1);

#ifdef FU_TRACE
  long long tr[32];
  int ntr = 0;
#define FU_T() do { if (rank == 0 && tid == 0 && ntr < 32) tr[ntr++] = clock64(); } while (0)
#else
#define FU_T() do { } while (0)
#endif
  int par = 0;           // parity of the current step: minibatch buffer, h_1 buffer, loss slots
  uint32_t step_no = 0;  // steps done: phase parity of the mbarriers
  float epoch_tot = 0.f;
  for (int ep = 0; ep < epochs; ++ep) {
    for (int st = 0; st < steps_per_epoch; ++st, par ^= 1, ++step_no) {
      const int s0 = st * a.batch;
      const int nb = min(a.batch, N - s0);
      int nst = st + 1, nep = ep;
      if (nst == steps_per_epoch) { nst = 0; ++nep; }
      const bool more = nep < epochs;
      if (more) index_stage(nep, nst);  // read by gather_async in the gradient phase
      const long long tm = run.t;  // the dropout masks' step: `iterations` before this step's increment
#ifdef FU_TRACE
      ntr = 0;
#endif
      FU_T();

      // ---- forward through the hidden layers: partial products, then reduce + activation + push ----
#pragma unroll
      for (int l = 0; l < ML; ++l) {
        if (l > L - 2) break;
        const int U = FU_U(l + 1);
        const float *A = sm + (l == 0 ? P.h0[par] : P.h[l][l == 1 ? par : 0]);
        const int act = d.act[l], outd = FU_DIM(l + 1);
        // this exchange's mbarrier: h_1 alternates between two buffers (one use every other step)
        const uint32_t bidx = 8u * (uint32_t)(2 * l + (l == 0 ? par : 0));
        const uint32_t bph = (l == 0 ? step_no >> 1 : step_no) & 1u;
        const uint32_t slice_bytes = (uint32_t)(U * SPP) * 4u;  // this layer's slice of one CTA: U rows, contiguous
        if (tid == 0) fu_bar_expect(bars + bidx, (FU_C - 1) * slice_bytes);
        if (warp < FU_KS)
          fu_partial(A, W + P.wc[l], fu_rk(FU_DIM(l)), U, SP, SPP, inv_nso, sm + P.scratch + warp * wstride, warp, lane);
        __syncthreads();
        FU_T();
        const float *bs = W + P.bs[l];
        float *Hn = sm + P.h[l + 1][l == 0 ? par : 0] + rank * U * SPP;  // own rows of h_{l+1}
        const bool drop = DROP && a.drop.rate[l] > 0.f;
        fu_reduce(sm + P.scratch, U, SP, inv_nq, wstride, [&](int u, int s, float4 sum) {
          if (rank * U + u < outd) {
            const float b = bs[u];
            float4 o = make_float4(act_fwd<EXT>(act, sum.x + b), act_fwd<EXT>(act, sum.y + b), act_fwd<EXT>(act, sum.z + b), act_fwd<EXT>(act, sum.w + b));
            if (drop) o = drop_fwd_unit4(a.drop, l, tm, s, rank * U + u, model, o);
            *reinterpret_cast<float4 *>(Hn + u * SPP + s) = o;
          }
        });
        if (warp < FU_KS || U * (SP >> 2) > 32 * FU_KS) fu_fence_async();  // the slice's writers: generic-proxy stores -> visible to the bulk-copy engine
        __syncthreads();   // slice complete (and the scratch is free for the next pass)
        if (tid < FU_C && tid != rank) {
          const uint32_t src = (uint32_t)__cvta_generic_to_shared(Hn);
          fu_bulk_push(fu_peer(Hn, tid), src, slice_bytes, fu_peer(sm + P.bars, tid) + bidx);
        }
        FU_T();
        fu_bar_wait(bars + bidx, bph);  // the other CTAs' slices of h_{l+1} have landed in THIS CTA's copy
        FU_T();
      }

      // ---- Dense(1) logit, loss, dL/dlogit: every CTA for itself ----
      const float *HLb = sm + P.h[L - 1][L - 1 == 1 ? par : 0];
      {
        const int kp = fdiv(tid, inv_sp), s = tid - kp * SP;
        if (kp < NLG) {
          float acc = 0.f;
          for (int k = kp; k < HL; k += NLG) acc = fmaf(HLb[k * SPP + s], W[P.wl + k], acc);
          sm[P.lg + kp * SP + s] = acc;
        }
      }
      __syncthreads();
      FU_T();
      const float inv_nb = 1.f / (float)nb;
      if (warp < 2) {  // SP <= 64: the samples sit in warps 0 and 1 (checked by the launcher)
        float dl = 0.f, lt = 0.f;
        if (tid < SP) {
          float u = W[P.bl];
          for (int kp = 0; kp < NLG; ++kp) u += sm[P.lg + kp * SP + tid];
          if (tid < nb) {
            const float zz = sm[P.zb + par * SP + tid];
            float g = stable_sigmoid(u) - zz;
            lt = fmaxf(u, 0.f) - u * zz + log1pf(expf(-fabsf(u)));
            if (WT) {
              const float ws = (wg ? sm[P.wb + tid] : 1.f) * (zz != 0.f ? a.fw.cw1 : a.fw.cw0);
              lt *= ws; g *= ws;
            }
            dl = g * inv_nb;
          }
          sm[P.dz + tid] = dl;
        }
        for (int o = 16; o > 0; o >>= 1) lt += __shfl_xor_sync(0xffffffffu, lt, o);
        if (lane == 0) sm[P.slots + 2 * par + warp] = lt;
      }

      // ---- optimizer scalars of this step ----
      FU_T();
      FU_T();
      const OptStep os = run.step(a.opt, a.sched);
      FU_T();
      __syncthreads();  // dz and the loss slots are in place
      FU_T();

      // ---- delta of the last hidden layer (elementwise, complete, every CTA) ----
      {
        float *DF = sm + (L - 1 >= 2 ? P.dg[L - 1] : P.dg[1]);
        const int nq = SP >> 2, actp = d.act[L - 2];
        const bool drop = DROP && a.drop.rate[L - 2] > 0.f;
        for (int e = tid; e < HL * nq; e += FU_THREADS) {
          const int k = fdiv(e, inv_nq), q = e - k * nq;
          const float4 hv = *reinterpret_cast<const float4 *>(HLb + k * SPP + 4 * q);
          const float4 dz = *reinterpret_cast<const float4 *>(sm + P.dz + 4 * q);
          const float w = W[P.wl + k];
          float4 o;
          if (drop) {
            o = drop_bwd_unit4<EXT>(a.drop, L - 2, tm, 4 * q, k, model, actp,
                                    make_float4(dz.x * w, dz.y * w, dz.z * w, dz.w * w), hv);
          } else {
            o.x = dz.x * w * act_bwd<EXT>(actp, hv.x);
            o.y = dz.y * w * act_bwd<EXT>(actp, hv.y);
            o.z = dz.z * w * act_bwd<EXT>(actp, hv.z);
            o.w = dz.w * w * act_bwd<EXT>(actp, hv.w);
          }
          *reinterpret_cast<float4 *>(DF + k * SPP + 4 * q) = o;
        }
      }
      __syncthreads();
      FU_T();

      // ---- reverse through the hidden layers: delta_i slice from delta_{i+1} and the row slice Wr_i ----
#pragma unroll
      for (int ii = 0; ii < ML; ++ii) {
        const int i = L - 2 - ii;
        if (i < 1) break;
        const int U = FU_U(i);
        const uint32_t bidx = 8u * (uint32_t)(2 * BORE_MAX_LAYERS + i);
        const int width = FU_DIM(i);
        const uint32_t slice_bytes = (uint32_t)(U * SPP) * 4u;
        if (i >= 2 && tid == 0) fu_bar_expect(bars + bidx, (FU_C - 1) * slice_bytes);
        if (warp < FU_KS)
          fu_partial(sm + P.dg[i + 1], W + P.wr[i], fu_rk(FU_DIM(i + 1)), U, SP, SPP, inv_nso,
                     sm + P.scratch + warp * wstride, warp, lane);
        __syncthreads();
        FU_T();
        const float *Hi = sm + P.h[i][i == 1 ? par : 0] + rank * U * SPP;  // own rows of h_i
        const int actp = d.act[i - 1];
        // delta_i slice: own rows of the complete buffer (i >= 2, pushed to the peers) or the local slice (i == 1)
        float *Dn = sm + (i >= 2 ? P.dg[i] + rank * U * SPP : P.d1);
        const bool drop = DROP && a.drop.rate[i - 1] > 0.f;  // h_i holds h~ of hidden layer i - 1
        fu_reduce(sm + P.scratch, U, SP, inv_nq, wstride, [&](int u, int s, float4 sum) {
          if (rank * U + u < width) {
            const float4 hv = *reinterpret_cast<const float4 *>(Hi + u * SPP + s);
            *reinterpret_cast<float4 *>(Dn + u * SPP + s) =
                drop ? drop_bwd_unit4<EXT>(a.drop, i - 1, tm, s, rank * U + u, model, actp, sum, hv)
                     : make_float4(sum.x * act_bwd<EXT>(actp, hv.x), sum.y * act_bwd<EXT>(actp, hv.y), sum.z * act_bwd<EXT>(actp, hv.z),
                                   sum.w * act_bwd<EXT>(actp, hv.w));
          }
        });
        if (i >= 2) {
          if (warp < FU_KS || U * (SP >> 2) > 32 * FU_KS) fu_fence_async();
          __syncthreads();
          if (tid < FU_C && tid != rank) {
            const uint32_t src = (uint32_t)__cvta_generic_to_shared(Dn);
            fu_bulk_push(fu_peer(Dn, tid), src, slice_bytes, fu_peer(sm + P.bars, tid) + bidx);
          }
          FU_T();
          fu_bar_wait(bars + bidx, step_no & 1u);
          FU_T();
        } else {
          __syncthreads();
          FU_T();
        }
      }

      // ---- weight gradients of the slices this CTA stores ----
      // Work items, one per thread (more than FU_THREADS: a second trip): 4 x 4 tiles of
      //   (a) the column copies Wc_l (rows: own units of layer l + 1, deltas; columns: units of layer l, h_l),
      //   (b) the row copies Wr_l (rows: own units of layer l, h_l; columns: units of layer l + 1, deltas),
      // then (c) single outputs: output-layer weights + bias (every CTA, identical) and the bias slices.
      // An item is decoded first (cheap, divergent) and computed after (convergent per kind); gradients go to
      // Gg (same index as the parameter), Adam follows for ALL parameters with every thread.
      const float *dzv = sm + P.dz;
      if (more) gather_async(par ^ 1, 0);  // next minibatch, in flight during this phase
      for (int item0 = 0; item0 < n_items; item0 += FU_THREADS) {
        const int item = item0 + tid;
        int kind = -1;  // 0 tile, 1 single output
        const float *Ab = nullptr, *Bb = nullptr;
        int RA = 1, Uc = 2, nta = 1, ta = 0, tu = 0, pbase = 0, wlimit = 0, kps = 0;
        int pi1 = 0;
        const int shalf = item >= n_tiles ? 1 : 0;
        if (item < 2 * n_tiles) {
          kind = 0;
          const int item = item0 + tid - shalf * n_tiles;  // the tile (shadows the work-item index)
          int base = 0;
          bool found = false;
#pragma unroll
          for (int blk = 0; blk < 2 * ML - 1; ++blk) {
            const bool colcopy = blk < ML;
            const int l = colcopy ? blk : blk - ML + 1;  // (a): l = 0..L-2, (b): l = 1..L-2
            if (l > L - 2 || found) continue;
            const int ra_ = colcopy ? FU_DIM(l) : FU_DIM(l + 1);
            const int u_ = colcopy ? FU_U(l + 1) : FU_U(l);
            const int nta_ = (ra_ + 3) >> 2, nt = nta_ * ((u_ + 3) >> 2);
            if (item < base + nt) {
              found = true;
              const int it = item - base;
              RA = ra_; Uc = u_; nta = nta_;
              tu = fdiv(it, 1.f / (float)nta); ta = it - tu * nta;
              kps = fu_kps(ra_);
              const float *hl = sm + (l == 0 ? P.h0[par] : P.h[l][l == 1 ? par : 0]);  // h_l
              // delta_{l+1}: complete buffer, or the local slice when it belongs to the first hidden layer of a
              // deeper net (only the column copy of W_0 reads that one)
              const bool dslice = (l + 1 == 1) && L > 2;
              const float *dn = sm + (dslice ? P.d1 : P.dg[l + 1]);
              if (colcopy) {
                Ab = hl;
                Bb = dn + (dslice ? 0 : rank * Uc * SPP);
                wlimit = FU_DIM(l + 1) - rank * Uc;
                pbase = P.wc[l];
              } else {
                Ab = dn;
                Bb = hl + rank * Uc * SPP;
                wlimit = FU_DIM(l) - rank * Uc;
                pbase = P.wr[l];
              }
              wlimit = min(wlimit, Uc);
            }
            base += nt;
          }
        } else if (item < n_items) {
          int k = item - 2 * n_tiles;
          if (k <= HL) {  // output layer: weights 0..HL-1, bias at HL
            kind = 1;
            Ab = k < HL ? HLb + k * SPP : nullptr;
            Bb = dzv;
            pi1 = P.wl + k;
          } else {
            k -= HL + 1;
            bool found = false;
#pragma unroll
            for (int l = 0; l < ML; ++l) {
              if (l > L - 2 || found) continue;
              const int u_ = FU_U(l + 1);
              if (k < u_) {
                found = true;
                if (rank * u_ + k < FU_DIM(l + 1)) {
                  kind = 1;
                  const bool dslice = (l + 1 == 1) && L > 2;
                  Bb = sm + (dslice ? P.d1 + k * SPP : P.dg[l + 1] + (rank * u_ + k) * SPP);
                  pi1 = P.bs[l] + k;
                }
              }
              k -= u_;
            }
          }
        }
        FU_T();
        if (kind == 0) {
          int ra[4];
          const float *ar[4], *br[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            ra[i] = min(ta + i * nta, RA - 1);
            ar[i] = Ab + ra[i] * SPP;
            br[i] = Bb + min(4 * tu + i, Uc - 1) * SPP;
          }
          float g[4][4];
          const int sh = (SP >> 1) & ~3;  // first half: [0, sh), second half: [sh, SP)
          fu_grad_tile(ar, br, shalf ? sh : 0, shalf ? SP : sh, g);
          FU_T();
          float *Go = Gg + shalf * P.npar;
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            if (4 * tu + e >= wlimit) continue;
#pragma unroll
            for (int i = 0; i < 4; ++i)
              if (ta + i * nta < RA) Go[pbase + (4 * tu + e) * kps + ra[i]] = g[e][i];
          }
        } else if (kind == 1) {
          Gg[pi1] = Ab ? fu_row_dot(Ab, Bb, SP) : fu_row_sum(Bb, SP);
        }
      }
      __syncthreads();  // gradients complete

      // ---- optimizer, in place, all parameters of this CTA (padding: zero gradient and slots, stays zero) ----
      float reg = 0.f;
      for (int pi = tid; pi < P.npar; pi += FU_THREADS) {
        float wv = W[pi], gg = Gg[pi] + Gg[P.npar + pi], m = Mm[pi], v = Vv[pi];
        if (a.any_reg) {
          // which block does pi belong to: l1 / l2 factors, and whether its term counts in the loss (every
          // parameter once: column copies and bias slices here, the output layer on rank 0).  The gradient
          // term goes on every copy and slice; padding (w = 0, g = 0) gets none, as sign(0) = 0.
          float l1 = 0.f, l2 = 0.f;
          bool cnt = false;
          if (pi >= P.wl) {
            if (pi < P.bl) { l1 = a.l1k[L - 1]; l2 = a.l2k[L - 1]; }
            else if (pi == P.bl) { l1 = a.l1b[L - 1]; l2 = a.l2b[L - 1]; }
            cnt = rank == 0;
          } else if (pi >= P.bs[0]) {
            for (int l = 0; l <= L - 2; ++l) if (pi >= P.bs[l]) { l1 = a.l1b[l]; l2 = a.l2b[l]; }
            cnt = true;
          } else if (L > 2 && pi >= P.wr[1]) {
            for (int l = 1; l <= L - 2; ++l) if (pi >= P.wr[l]) { l1 = a.l1k[l]; l2 = a.l2k[l]; }
          } else {
            for (int l = 0; l <= L - 2; ++l) if (pi >= P.wc[l]) { l1 = a.l1k[l]; l2 = a.l2k[l]; }
            cnt = true;
          }
          regularize(l1, l2, wv, reg, gg, cnt);
        }
        wv = opt_update<OPT>(a.opt, os, wv, gg, m, v);
        W[pi] = wv; Mm[pi] = m; Vv[pi] = v;
      }
      FU_T();
      if (rank == 0 && tid == 0) epoch_tot += (sm[P.slots + 2 * par] + sm[P.slots + 2 * par + 1]) * inv_nb * (float)nb;
      if (a.any_reg) {
        // regulariser terms: every CTA sums those of the parameters it owns (column copies, bias slices; rank 0
        // the output layer), rank 0 collects them after one cluster barrier (parity slots: the value is
        // overwritten two steps later, which no CTA reaches before rank 0 has passed the next barrier)
        reg = block_sum(reg, sm + P.scratch);
        if (tid == 0) sm[P.slots + 4 + par] = reg;
        fu_cluster_sync();
        if (rank == 0 && tid == 0) {
          float rg = 0.f;
          for (int c = 0; c < FU_C; ++c) rg += fu_ld(peer[c] + (uint32_t)(P.slots + 4 + par) * 4u);
          epoch_tot += rg * (float)nb;
        }
      }
      gather_wait();
      __syncthreads();  // weights updated, next minibatch in place
      FU_T();
#ifdef FU_TRACE
      if (rank == 0 && tid == 0 && (step_no == 200 || step_no == 201)) {
        printf("trace step %u:", step_no);
        for (int i = 1; i < ntr; ++i) printf(" %d", (int)(tr[i] - tr[i - 1]));
        printf(" | total %d\n", (int)(tr[ntr - 1] - tr[0]));
      }
#endif
    }
    if (rank == 0 && tid == 0 && a.loss_out) a.loss_out[pb.loss0 + ep] = epoch_tot / (float)N;
    epoch_tot = 0.f;
  }

  // ---- write back: the column copies partition W_l; rank 0 writes the output layer ----
  for (int l = 0; l <= L - 2; ++l) {
    const int in = d.dims[l], out = d.dims[l + 1], U = P.U[l + 1], kps = fu_kps(in);
    for (int e = tid; e < in * U; e += FU_THREADS) {
      const int k = e / U, u = e - k * U, j = rank * U + u;
      if (j < out) {
        const int gi = d.w_off[l] + k * out + j, pi = P.wc[l] + u * kps + k;
        gp[gi] = W[pi]; gm[gi] = Mm[pi]; gv[gi] = Vv[pi];
      }
    }
    for (int u = tid; u < U; u += FU_THREADS) {
      const int j = rank * U + u;
      if (j < out) {
        const int gi = d.b_off[l] + j;
        gp[gi] = W[P.bs[l] + u]; gm[gi] = Mm[P.bs[l] + u]; gv[gi] = Vv[P.bs[l] + u];
      }
    }
  }
  if (rank == 0) {
    const int hl = d.dims[L - 1];
    for (int k = tid; k <= hl; k += FU_THREADS) {
      const int gi = k < hl ? d.w_off[L - 1] + k : d.b_off[L - 1];
      gp[gi] = W[P.wl + k]; gm[gi] = Mm[P.wl + k]; gv[gi] = Vv[P.wl + k];
    }
    if (tid == 0) run.store(a.adam_t + model, a.opt_cache + model);
  }
  fu_cluster_sync();  // nobody exits while a peer may still address its shared memory
#undef FU_DIM
#undef FU_U
}

template <int NH, int HW, int SPT>
static int fu_launch(const FuArgs &a, int count, size_t smem, cudaStream_t stream) {
  const auto kern = with_build(opt_build(a.opt, a.sched), a.drop.any,
                               [](auto w, auto e, auto o, auto dr) { return fit_unit_kernel<NH, HW, SPT, w, e, o, dr>; },
                               a.fw.on, acts_ext(a.d.act, a.d.n_layers));
  BORE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<count * FU_C, FU_THREADS, smem, stream>>>(a);
  BORE_CUDA(cudaGetLastError());
  return 1;
}

}  // namespace

// The plan for a (padded) batch; false when the kernel does not take the net: no hidden layer, more
// than 64 samples (the loss reduction assumes the samples sit in two warps), or shared memory
static bool fu_plan(const MlpDesc &d, int batch, FuPlan &p, size_t &smem) {
  if (!make_fu_plan(d, batch, p)) return false;
  smem = (size_t)p.total * sizeof(float);
  return p.SP <= 64 && smem <= 226 * 1024;
}

int launch_fit_unit(const bore_mlp *h, const FitJob &job, int count, FitTable &tab, cudaStream_t stream) {
  FuArgs a{job};
  const int B = job.batch < job.N ? job.batch : job.N;
  // compile-time shapes: NH hidden layers of one width (16 / 32 / 64), padded batch 64; BORE_FIT_UNIT_GENERIC=1
  // forces the run-time-shape build (A/B timing, tests of both).  A smaller batch (the first iterations of a BO
  // run have fewer than 64 observations) is padded to 64 samples for them: zero rows, zero dL/dlogit.
  static const bool generic = [] { const char *e = getenv("BORE_FIT_UNIT_GENERIC"); return e && e[0] == '1'; }();
  const int nh = a.d.n_layers - 1, hw = a.d.n_layers >= 2 ? a.d.dims[1] : 0;
  bool uniform = a.d.n_layers >= 2;
  for (int i = 2; i <= nh; ++i) uniform = uniform && a.d.dims[i] == hw;
  const bool fixed_shape = !generic && uniform && B <= 64 &&
                           ((nh == 3 && (hw == 64 || hw == 32)) || (nh == 2 && (hw == 32 || hw == 16)));
  size_t smem;
  if (!fu_plan(a.d, fixed_shape ? 64 : B, a.P, smem)) return 0;
  BORE_CHECK_RC(tab.get(&a.probs));  // taken: the table goes up now
  if (fixed_shape) {
    if (nh == 3 && hw == 64) return fu_launch<3, 64, 64>(a, count, smem, stream);
    if (nh == 3 && hw == 32) return fu_launch<3, 32, 64>(a, count, smem, stream);
    if (nh == 2 && hw == 32) return fu_launch<2, 32, 64>(a, count, smem, stream);
    if (nh == 2 && hw == 16) return fu_launch<2, 16, 64>(a, count, smem, stream);
  }
  return fu_launch<0, 0, 0>(a, count, smem, stream);
}
