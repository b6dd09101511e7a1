// The job of an MLP fit launch and device helpers shared by the training kernels (fit.cu: FP32 FFMA;
// fit_unit.cu: FFMA2; fit_mma.cu: 3xTF32 tensor pipe).
#pragma once
#include "common.cuh"
#include "act.cuh"
#include "opt.cuh"
#include "dropout.cuh"

// What every MLP fit kernel reads besides its shared-memory plan: each kernel's arguments are a FitJob plus its
// plan (FitArgs, FitCArgs, FuArgs, FitMArgs).  The l1 / l2 factors are zero past the net's last layer.
// The build of a kernel (template flags OPT and DROP, with_build below): every optimizer but Adam and every
// learning-rate schedule run the OPT build.  fit_kernel (and lstm_fit_kernel) also run it for Adam when any_l1 is
// set, since their l1 terms are in the OPT build only; the cluster, unit-split and tensor-pipe kernels read l1 in
// every build.  Any dropout runs the build OPT = DROP = true, whatever the optimizer: the dropout code is in that
// build only, so the OPT build without dropout keeps its registers and instructions.
struct FitJob {
  MlpDesc d;
  float *params, *adam_m, *adam_v;
  long long *adam_t;
  int model0;
  const float *X, *z;
  int N, shared_data, batch, epochs;
  const int *perm;
  int shared_perm;
  const FitProblem *probs;  // NULL: uniform launch (fit_problem)
  float l2k[BORE_MAX_LAYERS], l2b[BORE_MAX_LAYERS];
  float l1k[BORE_MAX_LAYERS], l1b[BORE_MAX_LAYERS];
  int any_reg;  // some l1 or l2 factor is non-zero: the penalty is added to the reported loss
  int any_l1;   // some l1 factor is non-zero
  float *loss_out;
  OptHyper opt;
  FitWeights fw;
  float *opt_cache;  // [n_models] Nadam's momentum cache
  LrSchedule sched;
  Dropout drop;  // last: the members above keep their offsets
};

// The kernel of a fit launch: f(flags..., OPT, DROP) over the run-time flags bs, in one of the three builds that are
// instantiated -- (OPT = opt, DROP = false) without dropout, (true, true) with it (see FitJob).
template <class F, class... Bs>
auto with_build(bool opt, bool drop, F f, Bs... bs) {
  if (drop) return with_flags([&](auto... c) { return f(c..., std::true_type{}, std::true_type{}); }, bs...);
  return with_flags([&](auto... c) { return f(c..., std::false_type{}); }, bs..., opt);
}

// The launchers of the fit kernels, tried in this order by fit_run (fit.cu): 1 launched, 0 shape not taken (the
// next one is tried), < 0 error.  `tab`: the launch's problems (a ragged fit; job.N is then the largest N_p) or
// no table (uniform); a launcher uploads it after its last refusal.
// K1t (fit_mma.cu): tensor pipe, one CTA per model, on request only
int launch_fit_mma(const bore_mlp *h, const FitJob &job, int count, FitTable &tab, cudaStream_t stream);
// K1u (fit_unit.cu): one cluster per model, hidden units split over the CTAs
int launch_fit_unit(const bore_mlp *h, const FitJob &job, int count, FitTable &tab, cudaStream_t stream);

namespace {

__device__ __forceinline__ float stable_sigmoid(float u) {
  if (u >= 0.f) return 1.f / (1.f + expf(-u));
  const float e = expf(u);
  return e / (1.f + e);
}

__device__ __forceinline__ float block_sum(float v, float *red) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float t = 0.f;
  const int nw = blockDim.x >> 5;
  for (int i = 0; i < nw; ++i) t += red[i];
  return t;
}

// e / n for 0 <= e < 2^20 through a precomputed reciprocal (inv = 1.f / n): exact, the offset .5
// keeps the product away from integer boundaries
__device__ __forceinline__ int fdiv(int e, float inv) { return __float2int_rz(((float)e + 0.5f) * inv); }

}  // namespace
