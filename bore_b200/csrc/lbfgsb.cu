// K3: batched bound-constrained L-BFGS-B on device (sm_100a).
//
// Replaces the serial per-start scipy.optimize.minimize loop of bore/mixins.py:57-61.
// Structure: lock-step reverse communication, entirely on the device --
//
//     round r:   K2 (mlp_eval.cu) evaluates f,g for every start still asking for it, read
//                through a compacted active list;
//                the stepper consumes f,g and runs the L-BFGS-B state machine of
//                lbfgsb_core.h (Cauchy point, subspace minimisation, More'-Thuente line
//                search, BFGS update) for every active start until it either terminates or
//                posts its next trial point, appending itself to the next round's list.
//
// lbfgsb_warp_kernel: one WARP per active start, the start's state staged in shared memory
// (variant 1 of lbfgsb_core.h).  Finished starts drop out of the list, so late rounds cost
// only as much as the few starts that are still running (the per-start evaluation counts vary
// by >10x, SURVEY.md 7.2.3) -- and since such a round is a handful of warps, its cost is the
// LATENCY of one step, which is why a start gets a whole warp.  The host only polls the
// active counter, pipelined one chunk of rounds behind the launches.
//
// State.  Per start, a contiguous block in HBM: scalars (LbScal, 256 B) | xold gold d z (4n)
// | W = [Y S] (n x (2m+1)) | SY SS YY Tinv (4 m^2) doubles.  A step loads only what it
// touches: a step that just continues a line search reads the scalars and 4 vectors; the
// matrices are streamed into shared memory only when a new iteration starts, and written back
// only after a BFGS update.
//
// Tried and rejected (round 1, measured on B200, cfg 3): one THREAD per start with the state
// read in place from a structure-of-arrays block and the small dense scratch in local memory.
// Correct (same source compiled serially), but a heavy step is ~10^5 dependent instructions
// on L2-latency operands: 8-10 ms per round regardless of how many starts are active, against
// 4.7 ms for 65,536 starts with the warp kernel.  profiles/r01_notes.md has the launch list.
#include <float.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <cmath>

#include "common.cuh"
#include "lbfgsb_fused.h"
#include "lbfgsb_types.h"

namespace lbw {  // warp-collective variant, run-time history size m
#define LB_VARIANT 1
#include "lbfgsb_core.h"
#undef LB_VARIANT
}  // namespace lbw
namespace lbw10 {  // the same with m = 10 (SciPy's default maxcor) as a compile-time constant
#define LB_VARIANT 1
#define LB_MCONST 10
#include "lbfgsb_core.h"
#undef LB_MCONST
#undef LB_VARIANT
}  // namespace lbw10

// the two compilations of the core behind one name
template <int MC> struct LbCore;
template <> struct LbCore<0> {
  using Work = lbw::LbWork;
  static __device__ __forceinline__ void carve(Work &w, double *d, int *i, int n, int m) { lbw::lb_carve(w, d, i, n, m); }
  template <class Mem>
  static __device__ __forceinline__ int advance(const LbParams &P, Work &w, LbScal &s, Mem &mem, int stage) {
    return lbw::lb_advance(P, w, s, mem, stage);
  }
};
template <> struct LbCore<10> {
  using Work = lbw10::LbWork;
  static __device__ __forceinline__ void carve(Work &w, double *d, int *i, int n, int m) { lbw10::lb_carve(w, d, i, n, m); }
  template <class Mem>
  static __device__ __forceinline__ int advance(const LbParams &P, Work &w, LbScal &s, Mem &mem, int stage) {
    return lbw10::lb_advance(P, w, s, mem, stage);
  }
};
namespace {

constexpr int SCAL_BYTES = LB_SCAL_DOUBLES * sizeof(double);
static_assert(sizeof(LbScal) <= SCAL_BYTES, "LbScal grew past its slot");

struct LbLayout {
  // offsets in bytes from the workspace base
  size_t lo, hi, nbd, cnt, work, evals, lists, xf, f, g, pend, blocks, block_stride, total;
};

__host__ __device__ inline size_t align_up(size_t a, size_t b) { return (a + b - 1) / b * b; }

inline LbLayout make_layout(int S, int n, int m) {
  LbLayout L;
  size_t o = 0;
  L.lo = o; o += align_up(n * sizeof(double), 16);
  L.hi = o; o += align_up(n * sizeof(double), 16);
  L.nbd = o; o += align_up(n * sizeof(int), 16);
  L.cnt = o; o += 16;      // 3 rotating active counters (+pad)
  L.work = o; o += 16;     // 3 rotating work-queue heads (+pad)
  L.evals = o; o += 16;    // unsigned long long evals, bytes
  L.lists = o; o += align_up((size_t)2 * S * sizeof(int), 16);
  L.xf = o; o += align_up((size_t)S * n * sizeof(float), 16);
  L.f = o; o += align_up((size_t)S * sizeof(float), 16);
  L.g = o; o += align_up((size_t)S * n * sizeof(float), 16);
  L.pend = o; o += align_up((size_t)S * sizeof(int), 16);
  o = align_up(o, 256);
  L.block_stride = align_up((size_t)LB_PERSIST_DOUBLES(n, m) * sizeof(double), 128);
  L.blocks = o; o += L.block_stride * S;
  L.total = o;
  return L;
}

struct LbDev {
  LbParams P;
  int S;
  char *blocks;   // [S] per-start state blocks
  size_t block_stride;
  double *xreq;   // [S][n] last requested point (final x once a start is done)
  float *xf;      // [S][n] fp32 copy of the request for the MLP kernel (may be NULL)
  const void *F;  // [S]    objective values, indexed by start
  const void *G;  // [S][n] gradients
  int *lists;     // [2][S]
  int *cnt;       // [3]
  int *work;      // [3] work-queue heads: next unclaimed position of the round's active list
  unsigned long long *evals;
  unsigned long long *bytes;  // algorithmic bytes moved by the stepper (DESIGN.md, K3)
  int *pend;      // [S] (may be NULL)
};

__device__ __forceinline__ LbScal *scal_of(const LbDev &D, int sid) {
  return reinterpret_cast<LbScal *>(D.blocks + D.block_stride * sid);
}

// algorithmic bytes of one step (DESIGN.md, K3): what an ideal implementation has to move --
// scalars r+w, f, g and x read, the four vectors if a line search is in flight, the valid
// part of the limited memory when a new iteration starts, and what changed on the way out
__device__ __forceinline__ unsigned long long step_bytes(int n, int fg_size, bool was_ls,
                                                         bool heavy, int col_in, int col_out,
                                                         bool pend, bool updated) {
  unsigned long long b = 2ull * sizeof(LbScal) + (unsigned long long)fg_size * (1 + n) + 8ull * n;
  if (was_ls) b += 32ull * n;
  if (heavy && col_in > 0) b += 16ull * n * col_in + 32ull * col_in * col_in;
  b += pend ? 12ull * n : 8ull * n;
  if (heavy && pend) b += 32ull * n;
  if (updated) b += 16ull * n + 48ull * col_out + 8ull * col_out * col_out;
  return b;
}

// ---------------------------------------------------------------- init: one warp per start
__global__ void __launch_bounds__(128) lbfgsb_init_kernel(LbDev D, const double *__restrict__ X0) {
  const int n = D.P.n;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    D.cnt[0] = D.S; D.cnt[1] = 0; D.cnt[2] = 0;
    D.work[0] = 0; D.work[1] = 0; D.work[2] = 0;
    *D.evals = 0ULL;
    *D.bytes = 0ULL;
  }
  for (int sid = warp; sid < D.S; sid += nwarps) {
    for (int i = lane; i < n; i += 32) {
      double xi = X0[(size_t)sid * n + i];
      const int nb = D.P.nbd[i];
      if (nb > 0) {  // SciPy clips x0 into the box (_lbfgsb_py.py:359); `active` does the same
        if (nb <= 2 && xi <= D.P.lo[i]) xi = D.P.lo[i];
        else if (nb >= 2 && xi >= D.P.hi[i]) xi = D.P.hi[i];
      }
      D.xreq[(size_t)sid * n + i] = xi;
      if (D.xf) D.xf[(size_t)sid * n + i] = (float)xi;
    }
    if (lane == 0) {
      LbScal s;
      s.f = 0; s.fold = 0; s.theta = 1.0; s.gd = 0; s.gdold = 0; s.dtd = 0; s.dnorm = 0;
      s.stp = 0; s.stpmx = 0; s.sbgnrm = 0;
      s.finit = s.ginit = s.gtest = s.gx = s.gy = s.fx = s.fy = 0;
      s.stx = s.sty = s.stmin = s.stmax = s.width = s.width1 = 0;
      s.phase = LB_PH_START; s.col = 0; s.iupdat = 0; s.iter = 0; s.nit = 0;
      s.nfev = 1;  // the evaluation at x0
      s.ifun = 0; s.iback = 0; s.updatd = 0; s.status = -1; s.task = 0;
      s.brackt = 0; s.stage = 0; s.ls_task = LB_LS_START; s.nskip = 0; s.nintol = 0;
      s.resume = 0;
      *scal_of(D, sid) = s;
      D.lists[sid] = sid;
      if (D.pend) D.pend[sid] = 1;
    }
  }
}

// ---------------------------------------------------------------- warp variant: one round
// TMA bulk copies (cp.async.bulk, SASS UBLKCP) stage a start's persisted block between HBM and
// the warp's workspace: one instruction per direction instead of a load/store loop whose
// iterations each wait out an HBM round trip.
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "LB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra LB_DONE;\n"
      "bra LB_WAIT;\n"
      "LB_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst_smem)), "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void bulk_s2g(void *dst, const void *src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst),
               "r"(smem_u32(src_smem)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read() {  // source smem of all committed stores is free
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void bulk_wait_all() {  // all committed stores have landed
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}
__device__ __forceinline__ void bulk_prefetch_l2(const void *src, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void fence_async_smem() {  // generic-proxy smem writes -> async proxy
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// per-lane asynchronous copies (4 or 8 bytes: rows of any length and alignment), and the arrive on an
// mbarrier that fires once all of this lane's earlier copies have landed (.noinc: the barrier's
// expected count includes these arrivals)
template <int BYTES>
__device__ __forceinline__ void cp_async_g2s(void *dst_smem, const void *src) {
  static_assert(BYTES == 4 || BYTES == 8, "cp.async.ca copies 4, 8 or 16 bytes");
  asm volatile("cp.async.ca.shared.global [%0], [%1], %2;" ::"r"(smem_u32(dst_smem)), "l"(src), "n"(BYTES)
               : "memory");
}
__device__ __forceinline__ void cp_async_arrive(uint64_t *bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// Extra barriers per new iteration at which the warps of a CTA re-align (lb_advance's
// mem.phase()): at most 4 (before the Cauchy point, the K factorisation, the subspace
// minimisation and the line-search set-up).  Measured on B200, cfg 3 (stepper ms per step):
// free-running warps 148.7, rendezvous only 124.3, +1 barrier 124.5, +2 129.6, +3 131.4,
// +4 133.2 -- the default is the rendezvous alone (0); BORE_LB_NPHASE in the environment
// overrides it (-1 = free-running).
constexpr int LB_NPHASE_MAX = 4;

// A start's block is staged in two pieces: the prefix (scalars | t r d z) when the item is
// claimed -- together with the request x, the gradient row and f that its light stage reads, all on
// one mbarrier -- the limited-memory part (W and the m x m matrices, 87 % of the bytes) only when the
// light stage finds that a new iteration begins -- about half of all steps just continue a line
// search and never touch it.  The kernel requests the second piece right before the rendezvous
// (whose wait hides the latency); load() -- the hook lb_advance calls where the matrices are first
// needed -- waits for it.  The rest is bookkeeping of what has to be written back, and the phase
// barriers.
struct BlockMem {
  bool loaded = false, is_dirty = false, vec_dirty = false, requested = false;
  __device__ bool ld_kept() { return false; }  // the state was staged in from HBM: ld must be rebuilt
  int nph = 0, cap = LB_NPHASE_MAX;
  uint64_t *bar = nullptr;  // mbarrier of the second piece, and the parity of its current phase
  uint32_t parity = 0;
  __device__ void load() {
    if (!loaded && requested) { mbar_wait(bar, parity); __syncwarp(); }
    loaded = true;
  }
  __device__ void dirty() { is_dirty = true; }
  __device__ void dirty_vec() { vec_dirty = true; }
  // every warp of the CTA passes exactly `cap` of these per heavy pass (the kernel pads);
  // retries beyond that run unaligned
  __device__ void phase() {
    if (nph < cap) { __syncthreads(); ++nph; }
  }
};

// CTA header in dynamic shared memory: formk output map | lo | hi | nbd | two mbarriers per warp |
// two ints of the K-of-N rendezvous
__host__ __device__ inline size_t lb_header_bytes(int n, int wpb) {
  return align_up(LB_FORMK_ACC * 32 * sizeof(int), 16) + 2 * align_up(n * sizeof(double), 16) +
         align_up(n * sizeof(int), 16) + align_up(2 * wpb * sizeof(uint64_t) + 2 * sizeof(int), 16);
}

// One round.  Work items (positions of the round's active list) are claimed dynamically from a
// global queue head.  A warp runs the LIGHT stage of consecutive items (consume f,g, line-search
// logic, termination tests: small code, most often ending in the next trial point) until it
// holds an item that needs a new iteration; then all warps of the CTA meet and run the HEAVY
// stage (memory update, Cauchy point, K factorisation, subspace minimisation) phase by phase
// between CTA barriers -- ~10^4 instructions that the warps now fetch together instead of each
// thrashing the instruction caches from a different place (profiles/r01_notes.md).
template <typename FG, int MC>
__global__ void __maxnreg__(168) lbfgsb_warp_kernel(LbDev D, int round, size_t warp_bytes, int nphase, int kofn, int pf) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int n = D.P.n, m = D.P.m;
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int wpb = blockDim.x >> 5;
  const int cur = round % 3, nxt = (round + 1) % 3, clr = (round + 2) % 3;
  if (blockIdx.x == 0 && threadIdx.x == 0) { D.cnt[clr] = 0; D.work[clr] = 0; }
  const int n_active = D.cnt[cur];
  if (blockIdx.x * wpb >= n_active) return;
  const int *list_cur = D.lists + (size_t)(round & 1) * D.S;
  int *list_nxt = D.lists + (size_t)((round + 1) & 1) * D.S;
  int *qhead = D.work + cur;

  // ---- CTA header ----
  int *ftab = reinterpret_cast<int *>(smem_raw);
  double *s_lo = reinterpret_cast<double *>(smem_raw + align_up(LB_FORMK_ACC * 32 * sizeof(int), 16));
  double *s_hi = s_lo + align_up(n * sizeof(double), 16) / sizeof(double);
  int *s_nbd = reinterpret_cast<int *>(s_hi + align_up(n * sizeof(double), 16) / sizeof(double));
  uint64_t *bars = reinterpret_cast<uint64_t *>(reinterpret_cast<unsigned char *>(s_nbd) +
                                                align_up(n * sizeof(int), 16));
  uint64_t *bar = bars + 2 * wib, *bar2 = bar + 1;
  unsigned char *base = smem_raw + lb_header_bytes(n, wpb) + warp_bytes * wib;
  const uint32_t block_bytes = (uint32_t)(LB_PERSIST_DOUBLES(n, m) * sizeof(double));
  // first piece: scalars | t r d z; second piece: W and the matrices (both multiples of 16 bytes)
  const uint32_t p1_bytes = (uint32_t)(SCAL_BYTES + 4 * LB_NV(n) * sizeof(double));
  const uint32_t p2_bytes = block_bytes - p1_bytes;

  // K-of-N rendezvous (kofn > 0): the heavy stage starts as soon as ANY kofn warps of the CTA hold a
  // heavy item (named barrier 1 with a thread count), instead of waiting for the slowest of all of
  // them; warps that have run out of work keep feeding arrivals while somebody still waits.
  // (the two counters live behind the mbarriers in the CTA header: the kernel opts in to ALL of the
  // dynamic shared memory, which leaves no room for a static allocation)
  int &kn_wait = reinterpret_cast<int *>(bars + 2 * wpb)[0];
  int &kn_done = reinterpret_cast<int *>(bars + 2 * wpb)[1];
  if (threadIdx.x == 0) { kn_wait = 0; kn_done = 0; }
  // cur_i: the item whose block is staged (or on its way) in this warp's workspace, cur_sid its
  // start; nxt_i / nxt_sid: the one after it, claimed while cur_i runs and prefetched into L2
  // (a position >= n_active: the list is exhausted)
  int cur_i = 0;
  if (lane == 0) cur_i = atomicAdd(qhead, 1);
  cur_i = __shfl_sync(0xffffffffu, cur_i, 0);
  int cur_sid = cur_i < n_active ? list_cur[cur_i] : -1;
  if (lane == 0) {
    // the first piece's barrier completes on the bulk copy (one arrival with its byte count) and
    // on one cp.async arrival per lane (the light stage's x, g and f rows)
    mbar_init(bar, 1 + 32);
    mbar_init(bar2, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    if (cur_sid >= 0) {
      mbar_expect_tx(bar, p1_bytes);
      bulk_g2s(base, D.blocks + D.block_stride * cur_sid, p1_bytes, bar);
    }
  }
  int nxt_i = n_active, nxt_sid = -1;
#pragma unroll 1
  for (int o = threadIdx.x; o < LB_FORMK_ACC * 32; o += blockDim.x) ftab[o] = lbw::lb_formk_code(o, m);
#pragma unroll 1
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    s_lo[i] = D.P.lo[i];
    s_hi[i] = D.P.hi[i];
    s_nbd[i] = D.P.nbd[i];
  }
  __syncthreads();
  LbParams P = D.P;
  P.lo = s_lo; P.hi = s_hi; P.nbd = s_nbd;

  typename LbCore<MC>::Work w;
  LbCore<MC>::carve(w, reinterpret_cast<double *>(base),
                    reinterpret_cast<int *>(base + lbw::lb_work_doubles(n, m) * sizeof(double)), n, m);
  w.ftab = ftab;
  LbScal *s_smem = reinterpret_cast<LbScal *>(base);
  const FG *F = static_cast<const FG *>(D.F);
  const FG *G = static_cast<const FG *>(D.G);
  uint32_t parity = 0, parity2 = 0;
  unsigned long long my_bytes = 0, my_evals = 0;

  // The light stage's inputs of item `st`, copied asynchronously into the workspace: the request
  // x straight into w.x, the g row into w.g -- an fp32 row into its upper half, widened in place
  // once it has landed -- and f into w.q (scratch that nothing reads before the heavy stage).
  // Per-lane copies, so that a row of any length and alignment lands; each lane's arrival on `bar`
  // fires when its copies are done.  Callers order the workspace's earlier generic accesses first.
  const int g_off = sizeof(FG) == 4 ? LB_NV(n) : 0;  // in FG elements
  auto stage_light = [&](int st) {
    const double *xr = D.xreq + (size_t)st * n;
    const FG *gr = G + (size_t)st * n;
    FG *gs = reinterpret_cast<FG *>(w.g) + g_off;
#pragma unroll 1
    for (int i = lane; i < n; i += 32) {
      cp_async_g2s<8>(w.x + i, xr + i);
      cp_async_g2s<sizeof(FG)>(gs + i, gr + i);
    }
    if (lane == 31) cp_async_g2s<sizeof(FG)>(w.q, F + st);
    cp_async_arrive(bar);
  };
  if (cur_sid >= 0) stage_light(cur_sid);

  LbScal s;
  BlockMem mem;
  int sid = 0, col_in = 0;
  bool was_ls = false;

  // write an item back and put the next one on its way
  auto finish = [&](int pend) {
    // the slot in the next round's list: the atomic's result is used only after the stores below
    int pos = 0;
    if (pend && lane == 0) pos = atomicAdd(&D.cnt[nxt], 1);
    char *gblock = D.blocks + D.block_stride * sid;
    double *xr = D.xreq + (size_t)sid * n;
    if (mem.requested) {  // the second piece must have landed before its workspace is reused
      if (!mem.loaded) mbar_wait(bar2, parity2);
      parity2 ^= 1;
    }
    __syncwarp();
    my_bytes += step_bytes(n, (int)sizeof(FG), was_ls, mem.loaded, col_in, s.col, pend != 0, mem.is_dirty);
    if (pend) {
      float *xf = D.xf ? D.xf + (size_t)sid * n : nullptr;
#pragma unroll 1
      for (int i = lane; i < n; i += 32) {
        const double xi = w.x[i];
        xr[i] = xi;
        if (xf) xf[i] = (float)xi;
      }
      // a request equal to the point evaluated last is no new evaluation (SciPy memoises on x);
      // lb_advance has compared the two as it posted the request
      if (w.changed) s.nfev += 1;
    } else {
#pragma unroll 1
      for (int i = lane; i < n; i += 32) xr[i] = w.x[i];  // final iterate
    }
    // the head of the block that changed: scalars | t r d z | W and the matrices
    if (lane == 0) *s_smem = s;
    fence_async_smem();
    __syncwarp();
    cur_i = nxt_i;
    cur_sid = nxt_sid;
    // x, g and f of the next item lie outside the block, so they need not wait for the store below
    if (cur_sid >= 0) stage_light(cur_sid);
    if (lane == 0) {
      uint32_t bytes = SCAL_BYTES;
      if (pend && mem.vec_dirty) bytes += 4 * LB_NV(n) * sizeof(double);
      if (pend && mem.is_dirty) bytes = block_bytes;
      bulk_s2g(gblock, base, bytes);
      bulk_commit();
      if (pend) {
        list_nxt[pos] = sid;
        my_evals += 1;
      }
      if (D.pend) D.pend[sid] = pend;
      // the workspace may be overwritten once the store has read it
      bulk_wait_read();
      if (cur_sid >= 0) {
        mbar_expect_tx(bar, p1_bytes);
        bulk_g2s(base, D.blocks + D.block_stride * cur_sid, p1_bytes, bar);
      }
    }
    __syncwarp();
  };

#pragma unroll 1
  for (;;) {
    // ---- light stages until this warp holds an item that needs a new iteration ----
    bool holding = false;
#pragma unroll 1
    while (cur_i < n_active) {
      sid = cur_sid;
      // claim the item after this one; the claim's result is first needed once the light stage is done
      int claimed = 0;
      if (lane == 0) claimed = atomicAdd(qhead, 1);
#pragma unroll 1
      for (int i = lane; i < n; i += 32) {
        const int nb = s_nbd[i];
        w.iwhere[i] = nb == 0 ? -1 : ((nb == 2 && s_hi[i] - s_lo[i] <= 0.0) ? 3 : 0);
      }
      // the block's prefix, x, g and f (staged by the previous item's finish, or above)
      mbar_wait(bar, parity);
      parity ^= 1;
      __syncwarp();
      if (sizeof(FG) == 4) {
        // widen the fp32 row in place, 32 values at a time: a chunk's doubles overwrite only floats
        // of this chunk and of earlier ones, and every lane reads before any lane writes
        const float *gs = reinterpret_cast<const float *>(w.g) + g_off;
#pragma unroll 1
        for (int i0 = 0; i0 < n; i0 += 32) {
          const int i = i0 + lane;
          const float gi = i < n ? gs[i] : 0.f;
          __syncwarp();
          if (i < n) w.g[i] = (double)gi;
        }
        __syncwarp();
      }
      s = *s_smem;
      s.f = (double)*reinterpret_cast<const FG *>(w.q);
      __syncwarp();
      mem = BlockMem();
      mem.cap = nphase < 0 ? 0 : nphase;
      mem.bar = bar2;
      mem.parity = parity2;
      col_in = s.col;
      was_ls = s.phase == LB_PH_LNSRCH;
      const int r = LbCore<MC>::advance(P, w, s, mem, 1);
      // the item claimed above, and what its light stage reads pulled into L2 (the head of its
      // block, its request x, the g / f rows K2 wrote -- 0.9 GB of blocks stream through the 126 MB
      // L2 every round, so none of them would still be there): it is staged when this item finishes
      nxt_i = __shfl_sync(0xffffffffu, claimed, 0);
      nxt_sid = nxt_i < n_active ? list_cur[nxt_i] : -1;
      if (nxt_sid >= 0 && lane == 0) bulk_prefetch_l2(D.blocks + D.block_stride * nxt_sid, p1_bytes);
      if (nxt_sid >= 0 && pf) {
        const char *px = reinterpret_cast<const char *>(D.xreq + (size_t)nxt_sid * n);
        const char *pg = reinterpret_cast<const char *>(G + (size_t)nxt_sid * n);
        const int xb = n * (int)sizeof(double), gb = n * (int)sizeof(FG);
        const char *p = nullptr;
        if (lane < 16) { if (lane * 128 < xb) p = px + lane * 128; }
        else if (lane < 31) { if ((lane - 16) * 128 < gb) p = pg + (lane - 16) * 128; }
        else p = reinterpret_cast<const char *>(F + nxt_sid);
        if (p) asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
      }
      if (r == 2) {
        // a new iteration begins: request W and the matrices now, wait in mem.load()
        if (lane == 0) {
          mbar_expect_tx(bar2, p2_bytes);
          bulk_g2s(base + p1_bytes, D.blocks + D.block_stride * sid + p1_bytes, p2_bytes, bar2);
        }
        mem.requested = true;
        holding = true;
        break;
      }
      finish(r);
    }
    if (nphase < 0) {  // free-running warps (no alignment at all): tuning / comparison mode
      if (!holding) break;
      const int r = LbCore<MC>::advance(P, w, s, mem, 2);
      finish(r);
      continue;
    }
    if (kofn > 0) {
      if (!holding) break;  // the list is exhausted and nothing is in hand
      if (lane == 0) atomicAdd(&kn_wait, 1);
      __syncwarp();
      asm volatile("bar.sync 1, %0;" ::"r"(kofn * 32) : "memory");
      if (lane == 0) atomicSub(&kn_wait, 1);
      const int r = LbCore<MC>::advance(P, w, s, mem, 2);
      finish(r);
      continue;
    }
    if (!__syncthreads_or(holding ? 1 : 0)) break;
    // ---- heavy stage, phase-aligned across the CTA ----
    if (holding) {
      const int r = LbCore<MC>::advance(P, w, s, mem, 2);
#pragma unroll 1
      while (mem.nph < nphase) { __syncthreads(); ++mem.nph; }
      finish(r);
    } else {
#pragma unroll 1
      for (int k = 0; k < nphase; ++k) __syncthreads();
    }
  }
  if (lane == 0) {
    atomicAdd(D.bytes, my_bytes);
    atomicAdd(D.evals, my_evals);
    bulk_wait_all();
  }
  if (kofn > 0) {
    // out of work: feed the barrier while a warp of this CTA still waits for its group
    if (lane == 0) atomicAdd(&kn_done, 1);
#pragma unroll 1
    for (;;) {
      int done = 0, waiting = 0;
      if (lane == 0) {
        done = *reinterpret_cast<volatile int *>(&kn_done);
        waiting = *reinterpret_cast<volatile int *>(&kn_wait);
      }
      done = __shfl_sync(0xffffffffu, done, 0);
      waiting = __shfl_sync(0xffffffffu, waiting, 0);
      if (done >= wpb) break;
      if (waiting > 0) asm volatile("bar.arrive 1, %0;" ::"r"(kofn * 32) : "memory");
      __nanosleep(200);
    }
  }
}

__global__ void lbfgsb_results_kernel(LbDev D, double *x, double *fun, int *nit, int *nfev,
                                      int *status, int *task) {
  const int n = D.P.n;
  for (int sid = blockIdx.x * blockDim.x + threadIdx.x; sid < D.S; sid += gridDim.x * blockDim.x) {
    const LbScal *s = scal_of(D, sid);
    if (fun) fun[sid] = s->f;
    if (nit) nit[sid] = s->nit;
    if (nfev) nfev[sid] = s->nfev;
    if (status) status[sid] = s->status;
    if (task) task[sid] = s->task;
    if (x && x != D.xreq)
      for (int i = 0; i < n; ++i) x[(size_t)sid * n + i] = D.xreq[(size_t)sid * n + i];
  }
}

// ---------------------------------------------------------------- host side
// optional per-kernel timing of bore_lbfgsb_minimize (CUDA events on the launch stream)
struct LbProfile {
  bool enabled = false;
  std::vector<cudaEvent_t> pool;
  double k2_ms = 0, step_ms = 0, bytes = 0, evals = 0;
  int rounds = 0, k2_launches = 0, step_launches = 0;
  int fused = 0, grid = 0, block = 0;
  double tail_ms = 0;
  cudaEvent_t get(size_t i) {
    while (pool.size() <= i) {
      cudaEvent_t e;
      cudaEventCreate(&e);
      pool.push_back(e);
    }
    return pool[i];
  }
};
LbProfile g_prof;

struct StepLaunch {
  int grid, block;
  size_t warp_bytes, smem;
};

int plan_step(int S, int n, int m, int sm_count, StepLaunch &L) {
  L.warp_bytes = align_up(lbw::lb_work_doubles(n, m) * sizeof(double) + lbw::lb_work_ints(n) * sizeof(int), 16);
  const size_t hdr = lb_header_bytes(n, 12);
  const size_t max_block = 227 * 1024, max_sm = 228 * 1024;  // per CTA (opt-in) / per SM
  BORE_CHECK(L.warp_bytes + hdr <= max_block, "lbfgsb: n=%d needs %zu B of shared memory per start", n,
             L.warp_bytes + hdr);
  // warps per CTA: whatever packs the most starts into an SM's shared memory (the CTA header and
  // the 1 KB the system reserves per CTA are paid once per CTA); ties go to the larger CTA.
  // 168 registers per thread cap an SM at 12 warps.
  int wpb = 1, best = 0;
  for (int c = 1; c <= 12; ++c) {
    if (c * L.warp_bytes + hdr > max_block) break;
    int ctas = (int)(max_sm / (c * L.warp_bytes + hdr + 1024));
    if (ctas * c > 12) ctas = 12 / c;
    if (ctas * c >= best) { best = ctas * c; wpb = c; }
  }
  {  // tuning knob: warps per CTA (= size of the group that meets at the rendezvous)
    static int forced = -1;
    if (forced < 0) {
      const char *e = getenv("BORE_LB_WPB");
      forced = e ? atoi(e) : 0;
    }
    if (forced >= 1 && forced <= 12 && forced * L.warp_bytes + hdr <= max_block) wpb = forced;
  }
  L.block = wpb * 32;
  L.smem = hdr + wpb * L.warp_bytes;
  int per_sm = (int)(max_sm / (L.smem + 1024));
  if (per_sm * wpb > 12) per_sm = 12 / wpb;
  if (per_sm < 1) per_sm = 1;
  L.grid = sm_count * per_sm;
  const int need = (S + wpb - 1) / wpb;
  if (L.grid > need) L.grid = need;
  if (L.grid < 1) L.grid = 1;
  return 0;
}

// SciPy's bounds -> (l, u, nbd) (_lbfgsb_py.py:367-380), uploaded to lo_d / hi_d / nbd_d; fills P
int setup_problem(LbParams &P, double *lo_d, double *hi_d, int *nbd_d, int n, int m, const double *lo_h,
                  const double *hi_h, double ftol, double gtol, int maxiter, int maxfun, int maxls,
                  cudaStream_t stream) {
  std::vector<double> lo(n), hi(n);
  std::vector<int> nbd(n);
  int cnstnd = 0, boxed = 1;
  for (int i = 0; i < n; ++i) {
    const bool Lb = !isinf(lo_h[i]), Ub = !isinf(hi_h[i]);
    BORE_CHECK(!(Lb && Ub && lo_h[i] > hi_h[i]),
               "LBFGSB - one of the lower bounds is greater than an upper bound.");
    nbd[i] = Lb ? (Ub ? 2 : 1) : (Ub ? 3 : 0);
    lo[i] = Lb ? lo_h[i] : 0.0;
    hi[i] = Ub ? hi_h[i] : 0.0;
    if (nbd[i] != 2) boxed = 0;
    if (nbd[i] != 0) cnstnd = 1;
  }
  BORE_CUDA(cudaMemcpyAsync(lo_d, lo.data(), n * sizeof(double), cudaMemcpyHostToDevice, stream));
  BORE_CUDA(cudaMemcpyAsync(hi_d, hi.data(), n * sizeof(double), cudaMemcpyHostToDevice, stream));
  BORE_CUDA(cudaMemcpyAsync(nbd_d, nbd.data(), n * sizeof(int), cudaMemcpyHostToDevice, stream));
  BORE_CUDA(cudaStreamSynchronize(stream));  // the host vectors die at return
  P.n = n; P.m = m; P.maxiter = maxiter; P.maxfun = maxfun; P.maxls = maxls;
  P.cnstnd = cnstnd; P.boxed = boxed; P.ftol = ftol; P.pgtol = gtol;
  P.lo = lo_d; P.hi = hi_d; P.nbd = nbd_d;
  return 0;
}

int setup_params(LbDev &D, const LbLayout &L, char *work, int S, int n, int m, const double *lo_h,
                 const double *hi_h, double ftol, double gtol, int maxiter, int maxfun, int maxls,
                 cudaStream_t stream) {
  if (setup_problem(D.P, reinterpret_cast<double *>(work + L.lo), reinterpret_cast<double *>(work + L.hi),
                    reinterpret_cast<int *>(work + L.nbd), n, m, lo_h, hi_h, ftol, gtol, maxiter, maxfun,
                    maxls, stream))
    return -1;
  D.S = S;
  D.blocks = work + L.blocks;
  D.block_stride = L.block_stride;
  D.lists = reinterpret_cast<int *>(work + L.lists);
  D.cnt = reinterpret_cast<int *>(work + L.cnt);
  D.work = reinterpret_cast<int *>(work + L.work);
  D.evals = reinterpret_cast<unsigned long long *>(work + L.evals);
  D.bytes = D.evals + 1;
  return 0;
}

// one round of the stepper
template <typename FG, int MC>
int launch_round_mc(const LbDev &D, const StepLaunch &SL, int round, int nphase, cudaStream_t stream) {
  // opt in to > 48 KB of dynamic shared memory: the attribute belongs to the DEVICE's context,
  // so one flag per instantiation and device
  static bool attr_done[64] = {};
  int dev = 0;
  BORE_CUDA(cudaGetDevice(&dev));
  if (dev >= 64 || !attr_done[dev]) {
    BORE_CUDA(cudaFuncSetAttribute(lbfgsb_warp_kernel<FG, MC>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   227 * 1024));
    if (dev < 64) attr_done[dev] = true;
  }
  static int kofn = -1;
  if (kofn < 0) {
    const char *e = getenv("BORE_LB_KOFN");
    kofn = e ? atoi(e) : 0;
    if (kofn < 0) kofn = 0;
  }
  // (a group cannot be larger than the CTA; extra phase barriers and K-of-N do not mix)
  const int k_eff = (nphase == 0 && kofn > 0) ? std::min(kofn, SL.block / 32) : 0;
  static int pf = -1;
  if (pf < 0) {
    const char *e = getenv("BORE_LB_PREFETCH");
    pf = e ? atoi(e) : 1;
  }
  lbfgsb_warp_kernel<FG, MC><<<SL.grid, SL.block, SL.smem, stream>>>(D, round, SL.warp_bytes, nphase, k_eff, pf);
  BORE_CUDA(cudaGetLastError());
  return 0;
}

// one round of the stepper
template <typename FG>
int launch_round(const LbDev &D, const StepLaunch &SL, int round, cudaStream_t stream) {
  static int nphase = -1;
  if (nphase < 0) {
    const char *e = getenv("BORE_LB_NPHASE");
    nphase = e ? atoi(e) : 0;
    if (nphase < -1) nphase = -1;
    if (nphase > LB_NPHASE_MAX) nphase = LB_NPHASE_MAX;
  }
  if (D.P.m == 10) return launch_round_mc<FG, 10>(D, SL, round, nphase, stream);
  return launch_round_mc<FG, 0>(D, SL, round, nphase, stream);
}

// header kept at the very start of the external-API workspace so step/results can find things
struct ExtHeader {
  LbDev D;
  int round;
  int sm_count;
};
constexpr size_t EXT_HDR = 512;
static_assert(sizeof(ExtHeader) <= EXT_HDR, "ExtHeader too large");

int check_opts(int S, int D, int m, int maxls) {
  BORE_CHECK(S >= 1, "lbfgsb: S=%d", S);
  BORE_CHECK(D >= 1 && D <= BORE_MAX_DIM, "lbfgsb: D=%d outside [1,%d]", D, BORE_MAX_DIM);
  BORE_CHECK(m >= 1 && m <= BORE_LBFGSB_MAXCOR, "lbfgsb: maxcor=%d outside [1,%d]", m,
             BORE_LBFGSB_MAXCOR);
  BORE_CHECK(maxls > 0, "maxls must be positive.");
  return 0;
}

// BORE_LB_FUSED=0 in the environment sends bore_lbfgsb_minimize through the lock-step rounds
// (K2 launch + stepper launch per round) instead of the fused persistent kernel: the comparison
// arm of the tests and of tools/
// Which path runs a bore_lbfgsb_minimize call.  Measured on B200 (tools/fused_ab.py, cfg 3 net):
// the fused persistent kernel wins while the starts are few enough that the lock-step rounds run at
// their launch-latency floor -- 1,024 starts 1.7 vs 8.6 ms, 8,192 starts 23.9 vs 28.6 ms -- and
// loses at 65,536 (182 vs 130 ms): there the warps of an SM sit at nine different places of a
// ~100 KB instruction stream (ncu: no_instruction is 45 % of its stall cycles), which the
// rendezvous of the round kernel avoids.  Hence by default fused up to FUSED_MAX_STARTS starts,
// rounds above.  g_lb_mode: -1 from the environment (BORE_LB_FUSED = 0 never / 1 default / 2
// always fused when it fits), 0 default rule, 1 always rounds, 2 always fused.
// Re-measured in the third part of round 2 WITH the tail handover the default rule adds to the rounds (ms, fused vs
// rounds + handover): cfg-3 net (n = 50) 4,096 starts 13.8 vs 13.3, 6,144: 18.5 vs 17.6, 8,192: 24.1 vs 20.9, 10,240:
// 29.1 vs 23.8, 16,384: 45.9 vs 33.5; cfg-5 net (n = 8) 4,096: 3.1 vs 3.3, 8,192: 5.7 vs 6.7, 16,384: 10.9 vs 10.6;
// cfg-2 net (n = 6) 8,192: 7.1 vs 8.0, 16,384: 13.1 vs 13.0.  The heavy stage grows with n and with it the fetch
// problem of the fused kernel, so the limit is 4,096 starts (= the handover threshold: below it the rounds would
// hand everything over at once) for n > 16 and 16,384 for small problems.  BORE_LB_FUSED_MAX overrides it.
constexpr int FUSED_MAX_STARTS = 16384, FUSED_MAX_STARTS_LARGE_N = 4096, FUSED_LARGE_N = 16;
int g_lb_mode = -1;
int lb_mode() {
  if (g_lb_mode < 0) {
    const char *e = getenv("BORE_LB_FUSED");
    const int v = e ? atoi(e) : 1;
    g_lb_mode = v == 0 ? 1 : (v == 2 ? 2 : 0);
  }
  return g_lb_mode;
}
bool use_fused(const bore_mlp *h, int S, int m, int per_model) {
  const int mode = lb_mode();
  if (mode == 1) return false;
  // (batched problems: a few starts per model, the rounds never leave their latency floor)
  static const int fused_max_env = [] { const char *e = getenv("BORE_LB_FUSED_MAX"); return e ? atoi(e) : 0; }();
  const int fused_max = fused_max_env > 0 ? fused_max_env
                                          : (h->desc.dims[0] > FUSED_LARGE_N ? FUSED_MAX_STARTS_LARGE_N : FUSED_MAX_STARTS);
  if (mode == 0 && per_model == 0 && S > fused_max) return false;
  return m <= BORE_LBFGSB_MAXCOR && lbfgsb_fused_fits(h, m) != 0;
}

}  // namespace

extern "C" {

size_t bore_lbfgsb_workspace_bytes(int S, int D, int m) {
  if (S < 1 || D < 1 || m < 1) return 0;
  return EXT_HDR + make_layout(S, D, m).total;
}

int bore_lbfgsb_set_mode(int mode) {
  BORE_CHECK(mode >= 0 && mode <= 2, "bore_lbfgsb_set_mode: mode %d (0 default, 1 lock-step rounds, 2 fused)", mode);
  g_lb_mode = mode;
  return 0;
}

size_t bore_lbfgsb_minimize_workspace_bytes(const bore_mlp *h, int S, int m) {
  if (!h || S < 1 || m < 1) return 0;
  const int D = h->desc.dims[0];
  if (use_fused(h, S, m, 0)) return EXT_HDR + lbfgsb_fused_workspace_bytes(D);
  return bore_lbfgsb_workspace_bytes(S, D, m);
}

// shared body of bore_lbfgsb_minimize (n_models == 1, per_model == 0: all S starts belong to
// `model`) and bore_lbfgsb_minimize_multi (start i belongs to model model + i / per_model)
static int minimize_impl(bore_mlp *h, int model, int n_models, int per_model, int transform,
                         const double *X0_dev, int S, const double *lo_host, const double *hi_host,
                         int m, double ftol, double gtol, int maxiter, int maxfun, int maxls,
                         void *work_dev, size_t work_bytes, double *x_dev, double *fun_dev,
                         int32_t *nit_dev, int32_t *nfev_dev, int32_t *status_dev, int32_t *task_dev,
                         int *rounds_out, long long *evals_out, void *stream_) {
  BORE_NVTX("bore:argmax L-BFGS-B (K2+K3 / K3f)");
  BORE_CHECK(h != nullptr, "NULL handle");
  BORE_CHECK(model >= 0 && n_models >= 1 && model + n_models <= h->n_models,
             "models [%d,%d) outside [0,%d)", model, model + n_models, h->n_models);
  const int n = h->desc.dims[0];
  if (check_opts(S, n, m, maxls)) return -1;
  BORE_CHECK(transform >= 0 && transform <= BORE_TRANSFORM_EXP, "unknown transform code %d", transform);
  BORE_CHECK(x_dev && X0_dev && work_dev, "NULL buffer");
  BORE_CUDA(cudaSetDevice(h->device));
  cudaStream_t stream = (cudaStream_t)stream_;
  if (use_fused(h, S, m, per_model)) {
    // ---- the whole argmax in one persistent launch (lbfgsb_fused.cu) ----
    const size_t need = EXT_HDR + lbfgsb_fused_workspace_bytes(n);
    BORE_CHECK(work_bytes >= need, "lbfgsb workspace too small: %zu < %zu", work_bytes, need);
    char *work = static_cast<char *>(work_dev) + EXT_HDR;
    // [queue head, evaluation counter (64 B)] lo | hi | nbd
    double *lo_d = reinterpret_cast<double *>(work + 64);
    double *hi_d = lo_d + align_up(n * sizeof(double), 16) / sizeof(double);
    int *nbd_d = reinterpret_cast<int *>(hi_d + align_up(n * sizeof(double), 16) / sizeof(double));
    LbParams P;
    if (setup_problem(P, lo_d, hi_d, nbd_d, n, m, lo_host, hi_host, ftol, gtol, maxiter, maxfun, maxls, stream))
      return -1;
    if (g_prof.enabled) cudaEventRecord(g_prof.get(0), stream);
    long long evals = 0;
    FusedLaunchInfo info;
    const int rc = launch_lbfgsb_fused(h, model, n_models, per_model, transform, X0_dev, S, P, work, x_dev,
                                       fun_dev, nit_dev, nfev_dev, status_dev, task_dev, nullptr, &info, stream);
    if (rc) return rc;
    if (g_prof.enabled) cudaEventRecord(g_prof.get(1), stream);
    BORE_CUDA(cudaMemcpyAsync(&evals, work + 8, sizeof(evals), cudaMemcpyDeviceToHost, stream));
    cudaError_t e = cudaStreamSynchronize(stream);
    if (e != cudaSuccess) { bore_set_error("lbfgsb (fused): %s", cudaGetErrorString(e)); return -2; }
    if (evals_out) *evals_out = evals;
    if (rounds_out) *rounds_out = 1;
    if (g_prof.enabled) {
      float ms = 0;
      cudaEventElapsedTime(&ms, g_prof.get(0), g_prof.get(1));
      g_prof.k2_ms = 0; g_prof.step_ms = ms; g_prof.rounds = 1;
      g_prof.k2_launches = 0; g_prof.step_launches = 1;
      // HBM traffic an ideal implementation needs: start points in, iterates and 5 scalars out
      g_prof.bytes = (double)S * (16.0 * n + 24.0);
      g_prof.evals = (double)evals;
      g_prof.fused = 1; g_prof.grid = info.grid; g_prof.block = info.block;
    }
    return 0;
  }
  g_prof.fused = 0;
  const LbLayout L = make_layout(S, n, m);
  BORE_CHECK(work_bytes >= EXT_HDR + L.total, "lbfgsb workspace too small: %zu < %zu", work_bytes,
             EXT_HDR + L.total);
  char *work = static_cast<char *>(work_dev) + EXT_HDR;
  LbDev D;
  if (setup_params(D, L, work, S, n, m, lo_host, hi_host, ftol, gtol, maxiter, maxfun, maxls, stream))
    return -1;
  D.xreq = x_dev;
  D.xf = reinterpret_cast<float *>(work + L.xf);
  float *F = reinterpret_cast<float *>(work + L.f);
  float *G = reinterpret_cast<float *>(work + L.g);
  D.F = F; D.G = G;
  // batched problems: K2 finds each model's pending starts through per-start flags
  D.pend = per_model > 0 ? reinterpret_cast<int *>(work + L.pend) : nullptr;
  StepLaunch SL;
  if (plan_step(S, n, m, h->sm_count, SL)) return -1;
  {
    const int blocks = std::min((S + 3) / 4, h->sm_count * 8);
    lbfgsb_init_kernel<<<blocks, 128, 0, stream>>>(D, X0_dev);
    BORE_CUDA(cudaGetLastError());
  }
  // the weight image K2 stages from: packed once per call, not once per round
  if (mlp_eval_prepare(h, model, n_models, true, stream)) return -1;
  // pipelined polling: the active counter of chunk c is read while chunk c+1 is in flight
  const int CHUNK = 4;
  int *cnt_host = nullptr;
  BORE_CUDA(cudaMallocHost(&cnt_host, 2 * sizeof(int)));
  cudaEvent_t ev[2];
  BORE_CUDA(cudaEventCreateWithFlags(&ev[0], cudaEventDisableTiming));
  BORE_CUDA(cudaEventCreateWithFlags(&ev[1], cudaEventDisableTiming));
  int round = 0, rc = 0;
  // Tail handover: once few starts are still running, a lock-step round costs its launch-latency
  // floor (~93 us for K2 + stepper) whatever it does; the remaining starts are then finished by
  // the fused persistent kernel in resume mode (state blocks in, state blocks out) -- one launch in
  // which every start advances at the latency of its own steps.  BORE_LB_HANDOVER = the active
  // count at which to switch (0 = never).
  int handover = 0, handover_max = 0;
  if (per_model == 0 && lb_mode() != 1 && m <= BORE_LBFGSB_MAXCOR && lbfgsb_fused_fits(h, m)) {
    static int hmax = -1;
    if (hmax < 0) {
      const char *e = getenv("BORE_LB_HANDOVER");
      hmax = e ? atoi(e) : 4096;
      if (hmax < 0) hmax = 0;
    }
    handover_max = hmax;
  }
  bool have_prev = false;
  int slot = 0;
  const long long max_rounds = (long long)maxfun + (long long)maxls + 8;
  for (;;) {
    for (int k = 0; k < CHUNK; ++k, ++round) {
      const int *list = D.lists + (size_t)(round & 1) * S;
      if (g_prof.enabled) cudaEventRecord(g_prof.get(3 * (size_t)round), stream);
      rc = per_model > 0
               ? launch_mlp_eval_multi(h, model, n_models, per_model, true, transform, 1, D.xf, F, G,
                                       D.pend, stream, 1)
               : launch_mlp_eval(h, model, true, transform, 1, D.xf, S, F, G, list, D.cnt + round % 3,
                                 stream, 1);
      if (rc) break;
      if (g_prof.enabled) cudaEventRecord(g_prof.get(3 * (size_t)round + 1), stream);
      rc = launch_round<float>(D, SL, round, stream);
      if (rc) break;
      if (g_prof.enabled) cudaEventRecord(g_prof.get(3 * (size_t)round + 2), stream);
    }
    if (rc) break;
    if (cudaGetLastError() != cudaSuccess) { bore_set_error("lbfgsb stepper launch failed"); rc = -2; break; }
    cudaMemcpyAsync(&cnt_host[slot], D.cnt + round % 3, sizeof(int), cudaMemcpyDeviceToHost, stream);
    cudaEventRecord(ev[slot], stream);
    if (have_prev) {
      cudaError_t e = cudaEventSynchronize(ev[slot ^ 1]);
      if (e != cudaSuccess) { bore_set_error("lbfgsb: %s", cudaGetErrorString(e)); rc = -2; break; }
      if (cnt_host[slot ^ 1] == 0) break;
      if (handover_max > 0 && cnt_host[slot ^ 1] <= handover_max) { handover = cnt_host[slot ^ 1]; break; }
    }
    have_prev = true;
    slot ^= 1;
    if (round > max_rounds) { bore_set_error("lbfgsb: exceeded %lld rounds", max_rounds); rc = -3; break; }
  }
  float tail_ms = 0.f;
  if (!rc && handover > 0) {
    FusedResume R;
    R.list = D.lists + (size_t)(round & 1) * S;
    R.count = D.cnt + round % 3;
    R.blocks = D.blocks;
    R.block_stride = D.block_stride;
    R.qhead = D.work + 3;
    R.evals = D.evals;
    if (g_prof.enabled) cudaEventRecord(g_prof.get(3 * (size_t)round), stream);
    rc = launch_lbfgsb_fused(h, model, 1, 0, transform, nullptr, handover, D.P, work, D.xreq, nullptr, nullptr,
                             nullptr, nullptr, nullptr, nullptr, nullptr, stream, &R);
    if (g_prof.enabled) cudaEventRecord(g_prof.get(3 * (size_t)round + 1), stream);
  }
  if (!rc) {
    lbfgsb_results_kernel<<<std::min((S + 127) / 128, 1024), 128, 0, stream>>>(
        D, x_dev, fun_dev, nit_dev, nfev_dev, status_dev, task_dev);
    unsigned long long evals = 0;
    cudaMemcpyAsync(&evals, D.evals, sizeof(evals), cudaMemcpyDeviceToHost, stream);
    cudaError_t e = cudaStreamSynchronize(stream);
    if (e != cudaSuccess) { bore_set_error("lbfgsb: %s", cudaGetErrorString(e)); rc = -2; }
    // `evals` counts the requests posted after x0; add the S initial evaluations
    if (evals_out) *evals_out = (long long)evals + S;
    if (rounds_out) *rounds_out = round;
    if (g_prof.enabled && !rc) {
      unsigned long long bytes = 0;
      cudaMemcpy(&bytes, D.bytes, sizeof(bytes), cudaMemcpyDeviceToHost);
      g_prof.k2_ms = g_prof.step_ms = 0;
      for (int r = 0; r < round; ++r) {
        float a = 0, b = 0;
        cudaEventElapsedTime(&a, g_prof.get(3 * (size_t)r), g_prof.get(3 * (size_t)r + 1));
        cudaEventElapsedTime(&b, g_prof.get(3 * (size_t)r + 1), g_prof.get(3 * (size_t)r + 2));
        g_prof.k2_ms += a;
        g_prof.step_ms += b;
      }
      if (handover > 0) {  // the fused tail counts as stepper time (one more launch)
        cudaEventElapsedTime(&tail_ms, g_prof.get(3 * (size_t)round), g_prof.get(3 * (size_t)round + 1));
        g_prof.step_ms += tail_ms;
      }
      g_prof.tail_ms = tail_ms;
      g_prof.rounds = round;
      g_prof.k2_launches = g_prof.step_launches = round;
      g_prof.bytes = (double)bytes;
      g_prof.evals = (double)evals + S;
    }
  } else {
    cudaStreamSynchronize(stream);
  }
  cudaEventDestroy(ev[0]);
  cudaEventDestroy(ev[1]);
  cudaFreeHost(cnt_host);
  return rc;
}

int bore_lbfgsb_minimize(bore_mlp *h, int model, int transform, const double *X0_dev, int S,
                         const double *lo_host, const double *hi_host, int m, double ftol,
                         double gtol, int maxiter, int maxfun, int maxls, void *work_dev,
                         size_t work_bytes, double *x_dev, double *fun_dev, int32_t *nit_dev,
                         int32_t *nfev_dev, int32_t *status_dev, int32_t *task_dev, int *rounds_out,
                         long long *evals_out, void *stream_) {
  return minimize_impl(h, model, 1, 0, transform, X0_dev, S, lo_host, hi_host, m, ftol, gtol, maxiter,
                       maxfun, maxls, work_dev, work_bytes, x_dev, fun_dev, nit_dev, nfev_dev,
                       status_dev, task_dev, rounds_out, evals_out, stream_);
}

int bore_lbfgsb_minimize_multi(bore_mlp *h, int model0, int n_models, int starts_per_model,
                               int transform, const double *X0_dev, const double *lo_host,
                               const double *hi_host, int m, double ftol, double gtol, int maxiter,
                               int maxfun, int maxls, void *work_dev, size_t work_bytes,
                               double *x_dev, double *fun_dev, int32_t *nit_dev, int32_t *nfev_dev,
                               int32_t *status_dev, int32_t *task_dev, int *rounds_out,
                               long long *evals_out, void *stream_) {
  BORE_CHECK(starts_per_model >= 1 && starts_per_model <= 4096,
             "bore_lbfgsb_minimize_multi: starts_per_model=%d outside [1,4096]", starts_per_model);
  BORE_CHECK(n_models >= 1 && (long long)n_models * starts_per_model <= 0x7fffffffLL,
             "bore_lbfgsb_minimize_multi: n_models=%d", n_models);
  return minimize_impl(h, model0, n_models, starts_per_model, transform, X0_dev,
                       n_models * starts_per_model, lo_host, hi_host, m, ftol, gtol, maxiter, maxfun,
                       maxls, work_dev, work_bytes, x_dev, fun_dev, nit_dev, nfev_dev, status_dev,
                       task_dev, rounds_out, evals_out, stream_);
}

// per-kernel timing of the NEXT bore_lbfgsb_minimize calls (bench.py's roofline leg)
int bore_lbfgsb_profile(int enable) {
  g_prof.enabled = enable != 0;
  return 0;
}
// out[0] K2 total ms, out[1] stepper (or fused kernel) total ms, out[2] rounds (= launches of each
// kernel), out[3] algorithmic bytes, out[4] point evaluations, out[5] 1 = fused persistent kernel,
// out[6] / out[7] its grid / block size -- of the last profiled call
int bore_lbfgsb_last_profile(double *out) {
  BORE_CHECK(out != nullptr, "NULL argument");
  out[0] = g_prof.k2_ms; out[1] = g_prof.step_ms; out[2] = g_prof.rounds;
  out[3] = g_prof.bytes; out[4] = g_prof.evals;
  out[5] = g_prof.fused; out[6] = g_prof.grid; out[7] = g_prof.block;
  return 0;
}

// ---------------------------------------------------------------- reverse-communication API
int bore_lbfgsb_init(const double *X0_dev, int S, int n, const double *lo_host,
                     const double *hi_host, int m, double ftol, double gtol, int maxiter,
                     int maxfun, int maxls, void *work_dev, size_t work_bytes, double *xreq_dev,
                     int32_t *pend_dev, int device, void *stream_) {
  if (check_opts(S, n, m, maxls)) return -1;
  BORE_CHECK(X0_dev && work_dev && xreq_dev && pend_dev, "NULL buffer");
  BORE_CHECK(bore_device_count() > 0, "no CUDA device visible -- bore_b200 has no CPU fallback");
  BORE_CUDA(cudaSetDevice(device));
  cudaStream_t stream = (cudaStream_t)stream_;
  const LbLayout L = make_layout(S, n, m);
  BORE_CHECK(work_bytes >= EXT_HDR + L.total, "lbfgsb workspace too small: %zu < %zu", work_bytes,
             EXT_HDR + L.total);
  char *work = static_cast<char *>(work_dev) + EXT_HDR;
  ExtHeader H;
  memset(&H, 0, sizeof(H));
  if (setup_params(H.D, L, work, S, n, m, lo_host, hi_host, ftol, gtol, maxiter, maxfun, maxls, stream))
    return -1;
  H.D.xreq = xreq_dev;
  H.D.xf = nullptr;
  H.D.F = nullptr; H.D.G = nullptr;
  H.D.pend = pend_dev;
  H.round = 0;
  cudaDeviceProp prop;
  BORE_CUDA(cudaGetDeviceProperties(&prop, device));
  H.sm_count = prop.multiProcessorCount;
  const int blocks = std::min((S + 3) / 4, H.sm_count * 8);
  lbfgsb_init_kernel<<<blocks, 128, 0, stream>>>(H.D, X0_dev);
  BORE_CUDA(cudaGetLastError());
  BORE_CUDA(cudaMemcpyAsync(work_dev, &H, sizeof(H), cudaMemcpyHostToDevice, stream));
  BORE_CUDA(cudaStreamSynchronize(stream));
  return 0;
}

int bore_lbfgsb_step(const void *f_dev, const void *g_dev, int fg_is_f64, int S, int n,
                     void *work_dev, double *xreq_dev, int32_t *pend_dev, int *pending_out,
                     int device, void *stream_) {
  BORE_CHECK(f_dev && g_dev && work_dev, "NULL buffer");
  BORE_CUDA(cudaSetDevice(device));
  cudaStream_t stream = (cudaStream_t)stream_;
  ExtHeader H;
  BORE_CUDA(cudaMemcpyAsync(&H, work_dev, sizeof(H), cudaMemcpyDeviceToHost, stream));
  BORE_CUDA(cudaStreamSynchronize(stream));
  BORE_CHECK(H.D.S == S && H.D.P.n == n, "lbfgsb_step: workspace was initialised for S=%d D=%d",
             H.D.S, H.D.P.n);
  H.D.F = f_dev; H.D.G = g_dev;
  H.D.xreq = xreq_dev; H.D.pend = pend_dev;
  StepLaunch SL;
  if (plan_step(S, n, H.D.P.m, H.sm_count, SL)) return -1;
  const int rc = fg_is_f64 ? launch_round<double>(H.D, SL, H.round, stream)
                           : launch_round<float>(H.D, SL, H.round, stream);
  if (rc) return rc;
  BORE_CUDA(cudaGetLastError());
  H.round += 1;
  int pending = 0;
  BORE_CUDA(cudaMemcpyAsync(&pending, H.D.cnt + H.round % 3, sizeof(int), cudaMemcpyDeviceToHost, stream));
  BORE_CUDA(cudaMemcpyAsync(work_dev, &H, sizeof(H), cudaMemcpyHostToDevice, stream));
  BORE_CUDA(cudaStreamSynchronize(stream));
  if (pending_out) *pending_out = pending;
  return 0;
}

int bore_lbfgsb_results(int S, int n, void *work_dev, double *x_dev, double *fun_dev,
                        int32_t *nit_dev, int32_t *nfev_dev, int32_t *status_dev, int32_t *task_dev,
                        int device, void *stream_) {
  BORE_CHECK(work_dev, "NULL buffer");
  BORE_CUDA(cudaSetDevice(device));
  cudaStream_t stream = (cudaStream_t)stream_;
  ExtHeader H;
  BORE_CUDA(cudaMemcpyAsync(&H, work_dev, sizeof(H), cudaMemcpyDeviceToHost, stream));
  BORE_CUDA(cudaStreamSynchronize(stream));
  BORE_CHECK(H.D.S == S && H.D.P.n == n, "lbfgsb_results: workspace was initialised for S=%d D=%d",
             H.D.S, H.D.P.n);
  lbfgsb_results_kernel<<<std::min((S + 127) / 128, 1024), 128, 0, stream>>>(
      H.D, x_dev, fun_dev, nit_dev, nfev_dev, status_dev, task_dev);
  BORE_CUDA(cudaGetLastError());
  BORE_CUDA(cudaStreamSynchronize(stream));
  return 0;
}

}  // extern "C"
