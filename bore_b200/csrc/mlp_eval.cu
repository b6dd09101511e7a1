// K0 / K2: batched MLP forward and fused forward + reverse-through-input (sm_100a, FP32 FFMA).
//
// Replaces, for S points at once, what the reference evaluates one point per TensorFlow
// dispatch: keras predict (bore/mixins.py:50) and the value_and_gradient closure of
// convert() (bore/base.py:35-42, bore/decorators.py:48-65) with transform(-u)
// (bore/mixins.py:20).
//
// Mapping.  Weights are staged once per CTA into shared memory in ONE layout, W[k][j] with leading
// dimension (units rounded up to a chunk) + 4, zero-padded so that every inner loop is branch-free.
// The forward pass reads rows (a lane's 4 adjacent units: one LDS.128, lanes contiguous); the
// reverse pass reads the SAME image along j -- a lane owns input units ug, ug+UG, ug+2UG, ug+3UG of
// a chunk, so that the 8 lanes of a quarter-warp read 8 consecutive rows: stride LD = 4 (mod 32)
// words, 32 distinct banks per LDS.128.  (Round 1 kept a transposed copy for the reverse pass:
// 98 KB instead of 53 KB at Dense64x3, i.e. 11 instead of 14 resident warps per SM.)  Each WARP owns tiles of 16 points and carries them through
// all layers on its own: activations live in a per-warp shared-memory strip laid out
// [unit][point] (row stride 20 floats), so layers hand over with __syncwarp only -- no CTA
// barrier after the weight load.  Inside a tile every lane owns a 4-point x 4-unit
// register block: lane = pg*8 + ug, points pg*4..+3, units chunk*32 + ug*4..+3.  One k-step
// is two LDS.128 (4 activations, 4 weights) feeding 16 FFMA, so the loop is FFMA-issue
// bound, not shared-memory bound.  The reverse pass reuses the same loop on WT and
// multiplies by act'(h) (expressed through the stored layer output, as TF's *Grad kernels
// do) in the epilogue, overwriting the activation strip in place.
//
// Two lane mappings (template UGB): 8 unit-groups x 4 point-groups (tiles of 16 points, 32-unit
// chunks) for hidden widths <= 32, and 16 unit-groups x 2 point-groups (tiles of 8 points,
// 64-unit chunks) for wider layers -- the per-warp strip is half as large there, which doubles
// the warps that fit beside the weights in shared memory.
#include <algorithm>

#include <stdlib.h>

#include "common.cuh"
#include "act.cuh"

namespace {

template <int UGB>
struct Map {
  static constexpr int UG = 1 << UGB;        // lanes across units
  static constexpr int PG = 32 >> UGB;       // lanes across points
  static constexpr int TP = 4 * PG;          // points per warp tile
  static constexpr int CH = 4 * UG;          // units per chunk
  static constexpr int AST = TP + 4;         // activation strip row stride (floats)
};

struct SmemPlan {
  int wf[BORE_MAX_LAYERS];   // weights [inP][outP + 4] (rows >= in and columns >= out are zero)
  int bias[BORE_MAX_LAYERS]; // [outP]
  int wl;                    // final layer vector, padded
  int weights_total;         // floats
  int buf[BORE_MAX_LAYERS];  // per-warp strip offsets (floats, relative to the warp's base)
  int warp_total;            // floats per warp
  int wl_len;
};

__host__ __device__ inline int rup(int a, int b) { return (a + b - 1) / b * b; }

__host__ __device__ inline void make_plan(const MlpDesc &d, bool grad, int CH, int AST, SmemPlan &p) {
  int off = 0;
  const int G = d.n_layers - 1;  // GEMM (hidden) layers
  for (int l = 0; l < G; ++l) {
    int in = d.dims[l], out = d.dims[l + 1];
    // the reverse pass walks the rows of a whole chunk of input units: rows up to rup(in, CH)
    p.wf[l] = off; off += (grad ? rup(in, CH) : rup(in, 4)) * (rup(out, CH) + 4);
    p.bias[l] = off; off += rup(out, CH);
  }
  p.wl_len = G > 0 ? rup(d.dims[G], CH) : rup(d.dims[0], CH / 4);
  p.wl = off; off += p.wl_len;
  p.weights_total = rup(off, 4);
  int w = 0;
  p.buf[0] = 0; w += AST * (G > 0 ? rup(d.dims[0], 4) : p.wl_len);
  for (int l = 1; l <= G; ++l) { p.buf[l] = w; w += AST * rup(d.dims[l], CH); }
  p.warp_total = w;
}

// Packed FP32 FMA (sm_100a SASS FFMA2, PTX fma.rn.f32x2): two independent IEEE fp32 FMAs per lane and
// instruction -- the same roundings as two fmaf, so results do not change by a bit; what changes is
// the instruction count of a k-step (2 LDS.128 + 8 FFMA2 instead of 2 LDS.128 + 16 FFMA).  The pair
// (w, w) is folded by ptxas into the scalar-broadcast operand form (Rb.F32): no MOV is issued.
__device__ __forceinline__ uint64_t pk2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void fma2(uint64_t &c, uint64_t a, uint64_t b) {
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(c) : "l"(a), "l"(b));
}
__device__ __forceinline__ float2 upk2(uint64_t v) {
  float2 r;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(v));
  return r;
}

// acc[i][u] += sum_k A[k][pg*4+i] * W[k][col0+u],  k < K4 (multiple of 4)
template <int AST, bool F2>
__device__ __forceinline__ void tile_gemm(const float *__restrict__ A, const float *__restrict__ W,
                                          int K4, int ldw, float (&acc)[4][4]) {
  if (F2) {
    uint64_t c2[2][4];  // c2[h][u] = (acc[2h][u], acc[2h+1][u])
#pragma unroll
    for (int u = 0; u < 4; ++u) { c2[0][u] = pk2(acc[0][u], acc[1][u]); c2[1][u] = pk2(acc[2][u], acc[3][u]); }
#pragma unroll 2
    for (int k = 0; k < K4; k += 4) {
      float4 a[4], w[4];
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        a[kk] = *reinterpret_cast<const float4 *>(A + (k + kk) * AST);
        w[kk] = *reinterpret_cast<const float4 *>(W + (k + kk) * ldw);
      }
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        const uint64_t a01 = pk2(a[kk].x, a[kk].y), a23 = pk2(a[kk].z, a[kk].w);
        const float wv[4] = {w[kk].x, w[kk].y, w[kk].z, w[kk].w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const uint64_t ww = pk2(wv[u], wv[u]);
          fma2(c2[0][u], a01, ww);
          fma2(c2[1][u], a23, ww);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float2 lo = upk2(c2[0][u]), hi = upk2(c2[1][u]);
      acc[0][u] = lo.x; acc[1][u] = lo.y; acc[2][u] = hi.x; acc[3][u] = hi.y;
    }
    return;
  }
#pragma unroll 2
  for (int k = 0; k < K4; k += 4) {
    float4 a[4], w[4];
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      a[kk] = *reinterpret_cast<const float4 *>(A + (k + kk) * AST);
      w[kk] = *reinterpret_cast<const float4 *>(W + (k + kk) * ldw);
    }
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      const float av[4] = {a[kk].x, a[kk].y, a[kk].z, a[kk].w};
      const float wv[4] = {w[kk].x, w[kk].y, w[kk].z, w[kk].w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int u = 0; u < 4; ++u) acc[i][u] = fmaf(av[i], wv[u], acc[i][u]);
    }
  }
}

// Reverse pass on the forward image: acc[i][u] += sum_j A[j][pg*4+i] * W[row0 + u*RS][j],  j < J4
// (multiple of 4), in ascending j -- the same order and the same roundings as a k-loop over a
// transposed copy.  RS = lanes across units: unit u of this lane is row row0 + u*RS.
template <int AST, int RS, bool F2>
__device__ __forceinline__ void tile_gemm_T(const float *__restrict__ A, const float *__restrict__ Wrow,
                                            int J4, int ldw, float (&acc)[4][4]) {
  if (F2) {
    uint64_t c2[2][4];
#pragma unroll
    for (int u = 0; u < 4; ++u) { c2[0][u] = pk2(acc[0][u], acc[1][u]); c2[1][u] = pk2(acc[2][u], acc[3][u]); }
#pragma unroll 2
    for (int j = 0; j < J4; j += 4) {
      float4 a[4], w[4];
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) a[jj] = *reinterpret_cast<const float4 *>(A + (j + jj) * AST);
#pragma unroll
      for (int u = 0; u < 4; ++u) w[u] = *reinterpret_cast<const float4 *>(Wrow + u * RS * ldw + j);
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) {
        const uint64_t a01 = pk2(a[jj].x, a[jj].y), a23 = pk2(a[jj].z, a[jj].w);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float wv = jj == 0 ? w[u].x : jj == 1 ? w[u].y : jj == 2 ? w[u].z : w[u].w;
          const uint64_t ww = pk2(wv, wv);
          fma2(c2[0][u], a01, ww);
          fma2(c2[1][u], a23, ww);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float2 lo = upk2(c2[0][u]), hi = upk2(c2[1][u]);
      acc[0][u] = lo.x; acc[1][u] = lo.y; acc[2][u] = hi.x; acc[3][u] = hi.y;
    }
    return;
  }
#pragma unroll 2
  for (int j = 0; j < J4; j += 4) {
    float4 a[4], w[4];
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) a[jj] = *reinterpret_cast<const float4 *>(A + (j + jj) * AST);
#pragma unroll
    for (int u = 0; u < 4; ++u) w[u] = *reinterpret_cast<const float4 *>(Wrow + u * RS * ldw + j);
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
      const float av[4] = {a[jj].x, a[jj].y, a[jj].z, a[jj].w};
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float wv = jj == 0 ? w[u].x : jj == 1 ? w[u].y : jj == 2 ? w[u].z : w[u].w;
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[i][u] = fmaf(av[i], wv, acc[i][u]);
      }
    }
  }
}

// Writes one model's zero-padded weight image (the shared-memory plan of mlp_eval_kernel) to
// global memory: grid = models, launched once per parameter change instead of re-deriving the
// image in every CTA of every launch.
__global__ void __launch_bounds__(256)
mlp_pack_kernel(const MlpDesc d, const SmemPlan P, int CH, int grad, const float *__restrict__ params_all,
                float *__restrict__ packed_all) {
  const float *params = params_all + (size_t)blockIdx.x * d.n_params;
  float *out = packed_all + (size_t)blockIdx.x * P.weights_total;
  const int G = d.n_layers - 1;
  const int tid = threadIdx.x, nthr = blockDim.x;
  for (int l = 0; l < G; ++l) {
    const int in = d.dims[l], outd = d.dims[l + 1];
    const int rows = grad ? rup(in, CH) : rup(in, 4), outP = rup(outd, CH), ld = outP + 4;
    const float *Wg = params + d.w_off[l];
    float *wf = out + P.wf[l];
    for (int e = tid; e < rows * ld; e += nthr) {
      const int k = e / ld, j = e - k * ld;
      wf[e] = (k < in && j < outd) ? Wg[k * outd + j] : 0.f;
    }
    float *bs = out + P.bias[l];
    for (int e = tid; e < outP; e += nthr) bs[e] = e < outd ? params[d.b_off[l] + e] : 0.f;
  }
  {
    const int in = d.dims[G];
    float *wl = out + P.wl;
    for (int e = tid; e < P.weights_total - P.wl; e += nthr)
      wl[e] = e < in ? params[d.w_off[G] + e] : 0.f;  // incl. the pad up to weights_total
  }
}

__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

template <bool GRAD, int UGB, bool F2, bool EXT>
__global__ void __launch_bounds__(512)
mlp_eval_kernel(const MlpDesc d, const SmemPlan P, const float *__restrict__ params,
                const float *__restrict__ packed, const float *__restrict__ X,
                int S, const int *__restrict__ n_dev, const int *__restrict__ list,
                float *__restrict__ f_out, float *__restrict__ g_out, int transform, float sign,
                int per_model, const int *__restrict__ flags) {
  extern __shared__ __align__(128) float smem[];
  __shared__ __align__(8) uint64_t s_bar;
  using M = Map<UGB>;
  constexpr int TP = M::TP, AST = M::AST, CH = M::CH, UG = M::UG;
  const int G = d.n_layers - 1;
  const int tid = threadIdx.x, nthr = blockDim.x;
  // Two addressing modes.  Single model (per_model == 0): the launch covers S points (or the
  // first *n_dev of `list`), tiles are dealt round-robin to all warps of the grid.  Batched
  // problems (per_model > 0): CTA b works for model b on points [b*per_model, (b+1)*per_model),
  // of which only those with flags[point] != 0 are evaluated (flags == NULL: all of them).
  const bool multi = per_model > 0;
  int n, tile0, tile_step;
  long row_base = 0;
  int *llist = reinterpret_cast<int *>(smem + P.weights_total + (nthr >> 5) * P.warp_total);
  if (multi) {
    params += (size_t)blockIdx.x * d.n_params;
    packed += (size_t)blockIdx.x * P.weights_total;
    row_base = (long)blockIdx.x * per_model;
    if (flags) {  // order-preserving compaction of this model's pending starts
      __shared__ int s_cnt;
      if (tid == 0) s_cnt = 0;
      __syncthreads();
      for (int c0 = 0; c0 < per_model; c0 += nthr) {
        const int i = c0 + tid;
        const bool on = i < per_model && flags[row_base + i] != 0;
        const unsigned b = __ballot_sync(0xffffffffu, on);
        int wbase = 0;
        if ((tid & 31) == 0 && b) wbase = atomicAdd(&s_cnt, __popc(b));
        wbase = __shfl_sync(0xffffffffu, wbase, 0);
        if (on) llist[wbase + __popc(b & ((1u << (tid & 31)) - 1u))] = i;
      }
      __syncthreads();
      n = s_cnt;
      list = llist;
    } else {
      n = per_model;
      list = nullptr;
    }
    if (n == 0) return;
    tile0 = 0;
    tile_step = nthr >> 5;
  } else {
    // CTAs with no tile leave before paying for the weight staging: late L-BFGS-B rounds have
    // few active starts, and the launch is sized for all S of them
    n = n_dev ? min(*n_dev, S) : S;
    if (blockIdx.x * (nthr >> 5) * TP >= n) return;
    tile0 = blockIdx.x * (nthr >> 5);
    tile_step = gridDim.x * (nthr >> 5);
  }

  // ---- stage the pre-packed weight image: one TMA bulk copy (chunks of <= 64 KB) ----
  if (tid == 0) {
    const uint32_t bar = smem_addr(&s_bar);
    const uint32_t total = (uint32_t)P.weights_total * sizeof(float);
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(total) : "memory");
    for (uint32_t off = 0; off < total; off += 65536u) {
      const uint32_t nb = total - off < 65536u ? total - off : 65536u;
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   ::"r"(smem_addr(smem) + off), "l"(reinterpret_cast<const char *>(packed) + off), "r"(nb),
                     "r"(bar)
                   : "memory");
    }
  }
  __syncthreads();  // the barrier is initialised before anyone polls it
  {
    const uint32_t bar = smem_addr(&s_bar);
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "W_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], 0;\n"
        "@p bra W_DONE;\n"
        "bra W_WAIT;\n"
        "W_DONE:\n"
        "}\n" ::"r"(bar)
        : "memory");
  }
  const float b_last = params[d.b_off[G]];
  const int act_last = d.act[G];

  const int n_tiles = (n + TP - 1) / TP;
  const int warp = tid >> 5, lane = tid & 31, nwarps = nthr >> 5;
  const int ug = lane & (UG - 1), pg = lane >> UGB;
  float *strip = smem + P.weights_total + warp * P.warp_total;
  const int D = d.dims[0];
  const float *wl = smem + P.wl;

  for (int tile = tile0 + warp; tile < n_tiles; tile += tile_step) {
    const int p0 = tile * TP;
    // ---- load the 16 input rows, transposed into buf0[k][p] ----
    {
      float *xb = strip + P.buf[0];
      const int rows0 = G > 0 ? rup(D, 4) : P.wl_len;
      for (int pl = 0; pl < TP; ++pl) {
        const int idx = p0 + pl;
        const bool ok = idx < n;
        const long row = ok ? row_base + (list ? list[idx] : idx) : 0;
        for (int k = lane; k < rows0; k += 32)
          xb[k * AST + pl] = (ok && k < D) ? X[row * D + k] : 0.f;
      }
    }
    __syncwarp();

    // ---- forward through the hidden layers ----
    for (int l = 0; l < G; ++l) {
      const int in4 = rup(d.dims[l], 4), outP = rup(d.dims[l + 1], CH);
      const float *A = strip + P.buf[l] + pg * 4;
      float *H = strip + P.buf[l + 1];
      const float *W = smem + P.wf[l];
      const float *bs = smem + P.bias[l];
      const int a = d.act[l];
      for (int c = 0; c < outP; c += CH) {
        float acc[4][4] = {};
        tile_gemm<AST, F2>(A, W + c + ug * 4, in4, outP + 4, acc);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int unit = c + ug * 4 + u;
          const float b = bs[unit];
          float4 o;
          o.x = act_fwd<EXT>(a, acc[0][u] + b);
          o.y = act_fwd<EXT>(a, acc[1][u] + b);
          o.z = act_fwd<EXT>(a, acc[2][u] + b);
          o.w = act_fwd<EXT>(a, acc[3][u] + b);
          *reinterpret_cast<float4 *>(H + unit * AST + pg * 4) = o;
        }
      }
      __syncwarp();
    }

    // ---- final Dense(1): u = act(h . w + b) for this lane's 4 points ----
    float *HL = strip + P.buf[G];
    float up[4] = {0.f, 0.f, 0.f, 0.f};
    for (int k = ug; k < P.wl_len; k += UG) {
      const float4 hv = *reinterpret_cast<const float4 *>(HL + k * AST + pg * 4);
      const float w = wl[k];
      up[0] = fmaf(hv.x, w, up[0]);
      up[1] = fmaf(hv.y, w, up[1]);
      up[2] = fmaf(hv.z, w, up[2]);
      up[3] = fmaf(hv.w, w, up[3]);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
#pragma unroll
      for (int o = 1; o < UG; o <<= 1) up[i] += __shfl_xor_sync(0xffffffffu, up[i], o);
    }
    float dpre[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float u = act_fwd<EXT>(act_last, up[i] + b_last);
      float fval, dT;
      if (GRAD) {
        const float v = sign * u;
        if (transform == BORE_TRANSFORM_SIGMOID) {
          fval = 1.f / (1.f + expf(-v));
          dT = fval * (1.f - fval);
        } else if (transform == BORE_TRANSFORM_EXP) {
          fval = expf(v);
          dT = fval;
        } else {
          fval = v;
          dT = 1.f;
        }
        dpre[i] = dT * sign * act_bwd<EXT>(act_last, u);
      } else {
        fval = u;
      }
      const int idx = p0 + pg * 4 + i;
      if (ug == 0 && idx < n) f_out[row_base + (list ? list[idx] : idx)] = fval;
    }
    if (!GRAD) { __syncwarp(); continue; }

    // ---- reverse: delta of the last hidden layer (elementwise), then GEMMs on WT ----
    if (G == 0) {
      // no hidden layer: g = dpre * w
      for (int k = ug; k < D; k += UG) {
        const float w = wl[k];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int idx = p0 + pg * 4 + i;
          if (idx < n) g_out[(row_base + (list ? list[idx] : idx)) * D + k] = dpre[i] * w;
        }
      }
      __syncwarp();
      continue;
    }
    {
      const int a = d.act[G - 1];
      for (int k = ug; k < P.wl_len; k += UG) {
        float4 hv = *reinterpret_cast<const float4 *>(HL + k * AST + pg * 4);
        const float w = wl[k];
        hv.x = dpre[0] * w * act_bwd<EXT>(a, hv.x);
        hv.y = dpre[1] * w * act_bwd<EXT>(a, hv.y);
        hv.z = dpre[2] * w * act_bwd<EXT>(a, hv.z);
        hv.w = dpre[3] * w * act_bwd<EXT>(a, hv.w);
        *reinterpret_cast<float4 *>(HL + k * AST + pg * 4) = hv;
      }
    }
    __syncwarp();
    for (int l = G - 1; l >= 0; --l) {
      const int out4 = rup(d.dims[l + 1], 4), inP = rup(d.dims[l], CH), ldw = rup(d.dims[l + 1], CH) + 4;
      const float *A = strip + P.buf[l + 1] + pg * 4;   // delta_out [j][p]
      const float *W = smem + P.wf[l];                  // W [k][j]: rows = this layer's input units
      float *Hin = strip + P.buf[l];
      // this lane's units of a chunk: c + ug + UG*u (see the header: consecutive rows per quarter-warp)
      if (l > 0) {
        const int a = d.act[l - 1];
        for (int c = 0; c < inP; c += CH) {
          float acc[4][4] = {};
          tile_gemm_T<AST, UG, F2>(A, W + (c + ug) * ldw, out4, ldw, acc);
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            float *hp = Hin + (c + ug + UG * u) * AST + pg * 4;
            float4 hv = *reinterpret_cast<const float4 *>(hp);
            hv.x = acc[0][u] * act_bwd<EXT>(a, hv.x);
            hv.y = acc[1][u] * act_bwd<EXT>(a, hv.y);
            hv.z = acc[2][u] * act_bwd<EXT>(a, hv.z);
            hv.w = acc[3][u] * act_bwd<EXT>(a, hv.w);
            *reinterpret_cast<float4 *>(hp) = hv;
          }
        }
        __syncwarp();
      } else {
        // input gradient: stage through buf0 (x is dead) so the global store is coalesced
        for (int c = 0; c < inP; c += CH) {
          float acc[4][4] = {};
          tile_gemm_T<AST, UG, F2>(A, W + (c + ug) * ldw, out4, ldw, acc);
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int k = c + ug + UG * u;
            if (k < rup(D, 4))
              *reinterpret_cast<float4 *>(Hin + k * AST + pg * 4) =
                  make_float4(acc[0][u], acc[1][u], acc[2][u], acc[3][u]);
          }
        }
        __syncwarp();
        for (int pl = 0; pl < TP; ++pl) {
          const int idx = p0 + pl;
          if (idx >= n) break;
          const long row = row_base + (list ? list[idx] : idx);
          for (int k = lane; k < D; k += 32) g_out[row * D + k] = Hin[k * AST + pl];
        }
        __syncwarp();
      }
    }
  }
}

}  // namespace

static int variant_index(bool grad, int UGB) { return (grad ? 2 : 0) + (UGB == 4 ? 1 : 0); }

template <bool GRAD, int UGB>
static int pack_variant(const bore_mlp *h, int model0, int n_models, cudaStream_t stream) {
  using M = Map<UGB>;
  SmemPlan P;
  make_plan(h->desc, GRAD, M::CH, M::AST, P);
  const int v = variant_index(GRAD, UGB);
  MlpPackCache *pc = h->pack;
  BORE_CHECK(pc != nullptr, "handle has no pack cache");
  const size_t need = (size_t)h->n_models * P.weights_total;
  if (pc->cap[v] < need) {
    if (pc->buf[v]) BORE_CUDA(cudaFree(pc->buf[v]));
    pc->buf[v] = nullptr; pc->cap[v] = 0;
    BORE_CUDA(cudaMalloc(&pc->buf[v], need * sizeof(float)));
    pc->cap[v] = need;
  }
  mlp_pack_kernel<<<n_models, 256, 0, stream>>>(h->desc, P, M::CH, GRAD ? 1 : 0,
                                                 h->params + (size_t)model0 * h->desc.n_params,
                                                 pc->buf[v] + (size_t)model0 * P.weights_total);
  BORE_CUDA(cudaGetLastError());
  return 0;
}

constexpr int EVAL_MAX_SMEM = 227 * 1024;  // per CTA (opt-in)
constexpr int EVAL_STATIC_SMEM = 256;       // left for the kernel's static shared memory (mbarrier, counter, alignment)

// dynamic shared memory of an mlp_eval_kernel launch: the weight image, one activation strip per
// warp and, in batched mode with flags, the compacted start list
static size_t eval_smem_bytes(const SmemPlan &P, int warps, size_t list_bytes) {
  return (size_t)(P.weights_total + warps * P.warp_total) * sizeof(float) + list_bytes;
}

template <bool GRAD, int UGB>
static int launch_variant(const bore_mlp *h, const MlpDesc &d, int model0, const float *X,
                          int S, float *f, float *g, const int *list, const int *n_dev,
                          int transform, float sign, int n_models, int per_model, const int *flags,
                          int prepacked, cudaStream_t stream) {
  using M = Map<UGB>;
  SmemPlan P;
  make_plan(d, GRAD, M::CH, M::AST, P);
  const int max_smem = EVAL_MAX_SMEM;
  const bool multi = per_model > 0;
  const size_t list_bytes = (multi && flags) ? (size_t)per_model * sizeof(int) : 0;
  // warps per CTA: as many as fit (<= 16) -- in batched mode no more than the model has tiles
  int warps = 16;
  if (multi) warps = std::min(16, std::max(1, (per_model + M::TP - 1) / M::TP));
  while (warps > 1 && eval_smem_bytes(P, warps, list_bytes) + EVAL_STATIC_SMEM > (size_t)max_smem) --warps;
  const size_t smem = eval_smem_bytes(P, warps, list_bytes);
  BORE_CHECK(smem + EVAL_STATIC_SMEM <= (size_t)max_smem, "mlp_eval: model needs %zu B of shared memory (> %d)",
             smem + EVAL_STATIC_SMEM, max_smem);
  if (!prepacked && pack_variant<GRAD, UGB>(h, model0, n_models, stream)) return -1;
  const float *params = h->params + (size_t)model0 * d.n_params;
  const float *packed = h->pack->buf[variant_index(GRAD, UGB)] + (size_t)model0 * P.weights_total;
  int grid;
  if (multi) {
    grid = n_models;
  } else {
    const int n_tiles = (S + M::TP - 1) / M::TP;
    int ctas_needed = (n_tiles + warps - 1) / warps;
    int per_sm = (int)((size_t)max_smem / (smem + 1024));
    if (per_sm < 1) per_sm = 1;
    if (per_sm * warps > 48) per_sm = 48 / warps > 0 ? 48 / warps : 1;
    grid = h->sm_count * per_sm;
    if (grid > ctas_needed) grid = ctas_needed;
    if (grid < 1) grid = 1;
  }
  // packed FFMA2 inner loops unless BORE_K2_FFMA2=0 (the scalar-FFMA build stays for A/B timing; the
  // two give bit-identical results)
  static const bool f2 = [] { const char *e = getenv("BORE_K2_FFMA2"); return !(e && e[0] == '0'); }();
  const bool ext = acts_ext(d.act, d.n_layers);
  const auto kernel = f2 ? (ext ? mlp_eval_kernel<GRAD, UGB, true, true> : mlp_eval_kernel<GRAD, UGB, true, false>)
                         : (ext ? mlp_eval_kernel<GRAD, UGB, false, true> : mlp_eval_kernel<GRAD, UGB, false, false>);
  static bool attr_done[2][2][64] = {};  // per device: the attribute belongs to the device's context
  if (h->device >= 64 || !attr_done[f2][ext][h->device]) {
    BORE_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem - 256));
    if (h->device < 64) attr_done[f2][ext][h->device] = true;
  }
  kernel<<<grid, warps * 32, smem, stream>>>(d, P, params, packed, X, S, n_dev, list, f, g, transform, sign, per_model,
                                             flags);
  BORE_CUDA(cudaGetLastError());
  return 0;
}

static bool is_wide(const MlpDesc &d) {
  int widest = 0;
  for (int l = 1; l < d.n_layers; ++l) widest = d.dims[l] > widest ? d.dims[l] : widest;
  return widest > 32;  // 64-unit chunks, tiles of 8 points
}

static int dispatch(const bore_mlp *h, int model0, bool want_grad, int transform, int negate,
                    const float *X, int S, float *f, float *g, const int *list, const int *n_dev,
                    int n_models, int per_model, const int *flags, int prepacked, cudaStream_t stream) {
  const MlpDesc &d = h->desc;
  const bool wide = is_wide(d);
  const float sign = negate ? -1.f : 1.f;
#define BORE_EVAL(G_, U_)                                                                             \
  launch_variant<G_, U_>(h, d, model0, X, S, f, g, list, n_dev, transform, sign, n_models, per_model, \
                         flags, prepacked, stream)
  if (want_grad) return wide ? BORE_EVAL(true, 4) : BORE_EVAL(true, 3);
  return wide ? BORE_EVAL(false, 4) : BORE_EVAL(false, 3);
#undef BORE_EVAL
}

// bore_mlp_create: K0 and K2 must be able to stage the net with ONE warp (dispatch's variant, the
// plan and shared-memory sum of launch_variant); otherwise its first predict / argmax would fail
int mlp_eval_check_envelope(const MlpDesc &d) {
  const bool wide = is_wide(d);
  for (int grad = 0; grad < 2; ++grad) {
    SmemPlan P;
    if (wide) make_plan(d, grad != 0, Map<4>::CH, Map<4>::AST, P);
    else make_plan(d, grad != 0, Map<3>::CH, Map<3>::AST, P);
    const size_t need = eval_smem_bytes(P, 1, 0) + EVAL_STATIC_SMEM;
    BORE_CHECK(need <= (size_t)EVAL_MAX_SMEM,
               "bore_mlp_create: %s needs %zu B of shared memory for one warp (limit %d B)",
               grad ? "value and gradient (K2)" : "predict (K0)", need, EVAL_MAX_SMEM);
  }
  return 0;
}

int mlp_eval_prepare(const bore_mlp *h, int model0, int n_models, bool want_grad, cudaStream_t stream) {
  const bool wide = is_wide(h->desc);
  if (want_grad)
    return wide ? pack_variant<true, 4>(h, model0, n_models, stream)
                : pack_variant<true, 3>(h, model0, n_models, stream);
  return wide ? pack_variant<false, 4>(h, model0, n_models, stream)
              : pack_variant<false, 3>(h, model0, n_models, stream);
}

int launch_mlp_eval(const bore_mlp *h, int model, bool want_grad, int transform, int negate,
                    const float *X, int S, float *f, float *g, const int *list,
                    const int *n_dev, cudaStream_t stream, int prepacked) {
  if (S <= 0) return 0;
  return dispatch(h, model, want_grad, transform, negate, X, S, f, g, list, n_dev, 1, 0, nullptr,
                  prepacked, stream);
}

// batched problems: model model0+b evaluates points [b*per_model, (b+1)*per_model) of X (those
// with flags != 0 when `flags` is given), one CTA per model
int launch_mlp_eval_multi(const bore_mlp *h, int model0, int n_models, int per_model, bool want_grad,
                          int transform, int negate, const float *X, float *f, float *g,
                          const int *flags, cudaStream_t stream, int prepacked) {
  if (n_models <= 0 || per_model <= 0) return 0;
  return dispatch(h, model0, want_grad, transform, negate, X, n_models * per_model, f, g, nullptr,
                  nullptr, n_models, per_model, flags, prepacked, stream);
}
