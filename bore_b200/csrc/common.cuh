// Shared declarations for libbore_b200.so (sm_100a).  See include/bore_b200.h for the ABI.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>

#include "../../include/bore_b200.h"

// ---------------------------------------------------------------- error plumbing
void bore_set_error(const char *fmt, ...);

#define BORE_CHECK(cond, ...)            \
  do {                                   \
    if (!(cond)) {                       \
      bore_set_error(__VA_ARGS__);       \
      return -1;                         \
    }                                    \
  } while (0)

#define BORE_CUDA(call)                                                          \
  do {                                                                           \
    cudaError_t e__ = (call);                                                    \
    if (e__ != cudaSuccess) {                                                    \
      bore_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call,               \
                     cudaGetErrorString(e__));                                   \
      return -2;                                                                 \
    }                                                                            \
  } while (0)

// a call returning 0 or < 0 (error text already set): pass the error on
#define BORE_CHECK_RC(call)   \
  do {                        \
    const int rc__ = (call);  \
    if (rc__ != 0) return rc__; \
  } while (0)

// ---------------------------------------------------------------- NVTX ranges (SURVEY.md section 5)
// Header-only NVTX 3: a no-op unless a tool (nsys, ncu --nvtx) injects itself; no link dependency.
#include <nvtx3/nvToolsExt.h>
struct BoreNvtxRange {
  explicit BoreNvtxRange(const char *name) { nvtxRangePushA(name); }
  ~BoreNvtxRange() { nvtxRangePop(); }
};
#define BORE_NVTX(name) BoreNvtxRange bore_nvtx_range__(name)

// ---------------------------------------------------------------- model descriptor
// Passed by value to kernels (lives in kernel parameter space / constant bank).
struct MlpDesc {
  int n_layers;                     // Dense layers incl. the final (out_dim 1) layer
  int dims[BORE_MAX_LAYERS + 1];    // dims[0] = D
  int act[BORE_MAX_LAYERS];
  int w_off[BORE_MAX_LAYERS];       // offsets into the flat Keras-order parameter vector
  int b_off[BORE_MAX_LAYERS];
  int n_params;
};

// K0/K2 stage their weights from a pre-packed, zero-padded image (one per kernel variant:
// grad / no grad x narrow / wide lane mapping) with a single bulk copy; the cache is shared by
// shallow copies of the handle.
// Optimizer of a handle (bore_mlp_set_optimizer_kind / bore_lstm_set_optimizer_kind), passed by value to the fit
// kernels.  lr .. eps keep the places of Adam's former fields.
struct OptHyper {
  float lr;
  float b1;  // beta_1 (Adam, Adamax, Nadam) or rho (RMSprop, Adadelta)
  float b2;  // beta_2 (Adam, Adamax, Nadam)
  float eps;
  float momentum;  // RMSprop
  float init_acc;  // Adagrad's initial_accumulator_value
  int kind;        // BORE_OPT_*
  int centered;    // RMSprop
};

struct MlpPackCache {
  float *buf[4];
  size_t cap[4];  // floats allocated
};

struct bore_mlp {
  MlpDesc desc;
  MlpPackCache *pack;
  int n_models;
  int device;
  int sm_count;
  float *params;       // [n_models][n_params]
  float *adam_m;       // [n_models][n_params]
  float *adam_v;       // [n_models][n_params]
  long long *adam_t;   // [n_models]   Keras `iterations`
  float *opt_cache;    // [n_models]   Nadam's momentum cache
  OptHyper opt;
  float l2k[BORE_MAX_LAYERS], l2b[BORE_MAX_LAYERS];  // l2 regularisers per layer
  int fit_mode;  // 0 auto, 1 one CTA per model (FFMA), 2 one cluster per model, samples split (FFMA), 3 tensor
                 // pipe, 4 one cluster per model, units split (FFMA2)  (bore_mlp_set_fit_mode)
  void *tab_pinned;      // pinned staging buffer of the ragged fit's problem table (FitTable), tab_cap bytes
  size_t tab_cap;
  cudaEvent_t tab_done;  // recorded behind the last copy out of tab_pinned
};

static inline int round_up(int a, int b) { return (a + b - 1) / b * b; }

// Per-sample loss weights of a weighted fit / evaluate (bore_mlp_fit_weighted): the weight of sample i is
// w[i] (1 when w is NULL) times cw1 if its label is 1, else cw0.  w has the layout of the labels.  on == 0:
// unweighted, the kernels run the arithmetic of bore_mlp_fit unchanged.
struct FitWeights {
  const float *w;
  float cw0, cw1;
  int on;
};

// One problem of a fit launch, read by its CTA (or cluster) at entry: the model it trains, the first of its
// rows of X / z / w, of its permutation entries ([epochs][N] from there) and of its epoch losses, and its
// observation count and epochs.  bore_mlp_fit_ragged passes a device table of them in launch order; the
// uniform entry points pass none and every problem is derived from the launch's scalars (fit_problem).
struct FitProblem {
  long long row0, perm0, loss0;
  int model, N, epochs, pad_;
};

#ifdef __CUDACC__
// the loss weight of one sample (device code; row >= 0)
__device__ __forceinline__ float fit_sample_weight(const FitWeights &fw, const float *w, int row, float z) {
  return (w ? w[row] : 1.f) * (z != 0.f ? fw.cw1 : fw.cw0);
}

// problem `b` of a uniform launch whose arguments `a` carry model0 / N / epochs / shared_data / shared_perm
template <class A>
__device__ __forceinline__ FitProblem fit_problem_uniform(const A &a, int b) {
  FitProblem p;
  p.model = a.model0 + b;
  p.N = a.N;
  p.epochs = a.epochs;
  p.row0 = a.shared_data ? 0 : (long long)b * a.N;
  p.perm0 = a.shared_perm ? 0 : (long long)b * a.epochs * a.N;
  p.loss0 = (long long)b * a.epochs;
  p.pad_ = 0;
  return p;
}
// problem `b` of any launch: from the table a.probs when there is one
template <class A>
__device__ __forceinline__ FitProblem fit_problem(const A &a, int b) {
  return a.probs ? a.probs[b] : fit_problem_uniform(a, b);
}
#endif

// A small host table for one launch, copied to the device on the launch's stream (cudaMallocAsync, plain
// cudaMemcpyAsync) and freed on that stream when the object goes out of scope, i.e. after every launch
// enqueued before: a later call never overwrites a table an earlier launch may still read.
struct StreamTable {
  void *dev = nullptr;
  cudaStream_t stream = nullptr;
  cudaError_t upload(const void *host, size_t bytes, cudaStream_t s) {
    stream = s;
    cudaError_t e = cudaMallocAsync(&dev, bytes, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dev, host, bytes, cudaMemcpyHostToDevice, s);
    return e;
  }
  ~StreamTable() {
    if (dev) cudaFreeAsync(dev, stream);
  }
};

// The problem table of a ragged fit (FitProblem, launch order) on its way to the device.  get() stages it through
// the handle's pinned buffer (so that the copy is asynchronous) into a StreamTable on the launch's stream; the
// launchers call it after their last refusal, right before the launch, so that a refused call enqueues nothing.
// A uniform fit has no table: host == NULL, get() gives NULL.
struct FitTable {
  bore_mlp *h;
  const FitProblem *host;
  int n;
  cudaStream_t stream;
  StreamTable dev;
  int get(const FitProblem **out);  // 0, or < 0 with the error text set
};

// ---------------------------------------------------------------- optimizer state
// Slot 0, slot 1, `iterations` and the Nadam cache of `count` consecutive models, set to the initial values of
// the kind (opt.init_acc for Adagrad's accumulator, 1 for the cache, zeros else) on `stream`.
int opt_reset_state(const OptHyper &opt, float *s0, float *s1, size_t n_params, long long *t_dev, float *cache,
                    int count, cudaStream_t stream);
// bore_*_set_optimizer_kind's check of (kind, hp); 0, or -1 with the error text set
int opt_from_array(int kind, const float *hp, OptHyper &out, const char *who);

// ---------------------------------------------------------------- launchers (one per .cu)
// K0 / K2.  `list` (may be NULL) is a device array of row indices: point i of the launch
// is row list[i] of X / f / g (used by the L-BFGS-B driver's compacted active list);
// `n_dev` (may be NULL) is a device int holding the number of points (<= S).
// `prepacked` != 0: the caller has run mlp_eval_prepare for these models since the parameters
// last changed (the L-BFGS-B driver packs once per call, not once per round).
int launch_mlp_eval(const bore_mlp *h, int model, bool want_grad, int transform, int negate,
                    const float *X, int S, float *f, float *g, const int *list,
                    const int *n_dev, cudaStream_t stream, int prepacked = 0);
int mlp_eval_prepare(const bore_mlp *h, int model0, int n_models, bool want_grad, cudaStream_t stream);
// batched problems (BASELINE.json configs[3]): one CTA per model; model model0+b owns points
// [b*per_model, (b+1)*per_model) of X / f / g; `flags` (may be NULL) selects the points to do.
int launch_mlp_eval_multi(const bore_mlp *h, int model0, int n_models, int per_model, bool want_grad,
                          int transform, int negate, const float *X, float *f, float *g,
                          const int *flags, cudaStream_t stream, int prepacked = 0);
// bore_mlp_create's check of a net against the kernels' shared-memory plans (mlp_eval.cu, fit.cu): 0 when
// it runs, else -1 with the shared memory needed and the limit in the error text.  Host only, no device.
int mlp_eval_check_envelope(const MlpDesc &d);
int fit_check_envelope(const MlpDesc &d);
// K1t (fit_mma.cu): 1 launched, 0 shape not taken (caller falls back to the FFMA kernels), < 0 error.
// `tab`: the launch's problems (a ragged fit; N is then the largest N_p) or no table (uniform).
int launch_fit_mma(const bore_mlp *h, int model0, int count, const float *X_dev, const float *z_dev, int N,
                   int shared_data, int batch_size, int epochs, const int32_t *perm_dev, int shared_perm,
                   float *loss_out_dev, const FitWeights &fw, FitTable &tab, cudaStream_t stream);
// K1u (fit_unit.cu): one cluster per model, hidden units split over the CTAs.  1 launched, 0 shape not
// taken (caller falls back to the sample-split cluster kernel), < 0 error
int launch_fit_unit(const bore_mlp *h, int model0, int count, const float *X_dev, const float *z_dev, int N,
                    int shared_data, int batch_size, int epochs, const int32_t *perm_dev, int shared_perm,
                    float *loss_out_dev, const FitWeights &fw, FitTable &tab, cudaStream_t stream);
