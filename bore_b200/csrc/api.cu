// C-ABI glue of libbore_b200.so: handle management, error text, parameter I/O, and the
// FP32 FFMA peak microbenchmark.  See include/bore_b200.h.
#include <stdarg.h>
#include <string.h>

#include "common.cuh"

static thread_local char g_err[1024] = "";

void bore_set_error(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// ---------------------------------------------------------------- optimizer state
__global__ void fill_kernel(float *p, size_t n, float v) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}

// v = 0 is a memset (the only path Adam takes); other values (Adagrad's initial accumulator, Nadam's cache
// of 1) are no byte pattern and need the fill kernel
static int fill_async(float *p, size_t n, float v, cudaStream_t st) {
  if (v == 0.f) {
    BORE_CUDA(cudaMemsetAsync(p, 0, n * sizeof(float), st));
  } else {
    const size_t blocks = (n + 255) / 256;
    fill_kernel<<<(unsigned)(blocks < 1024 ? blocks : 1024), 256, 0, st>>>(p, n, v);
    BORE_CUDA(cudaGetLastError());
  }
  return 0;
}

int opt_reset_state(const OptHyper &opt, float *s0, float *s1, size_t n_params, long long *t_dev, float *cache,
                    int count, cudaStream_t st) {
  const size_t n = (size_t)count * n_params;
  BORE_CHECK_RC(fill_async(s0, n, opt.kind == BORE_OPT_ADAGRAD ? opt.init_acc : 0.f, st));
  BORE_CUDA(cudaMemsetAsync(s1, 0, n * sizeof(float), st));
  if (t_dev) BORE_CUDA(cudaMemsetAsync(t_dev, 0, count * sizeof(long long), st));
  if (opt.kind != BORE_OPT_ADAM) BORE_CHECK_RC(fill_async(cache, count, 1.f, st));
  return 0;
}

int opt_from_array(int kind, const float *hp, OptHyper &o, const char *who) {
  BORE_CHECK(kind >= BORE_OPT_ADAM && kind <= BORE_OPT_NADAM,
             "%s: unknown optimizer kind %d (BORE_OPT_ADAM .. BORE_OPT_NADAM; SGD and Ftrl have no kernel)", who, kind);
  BORE_CHECK(hp != nullptr, "%s: hyper-parameter array is NULL", who);
  o = OptHyper{hp[0], hp[1], hp[2], hp[3], hp[4], hp[5], kind, hp[6] != 0.f};
  const bool rho = kind == BORE_OPT_RMSPROP || kind == BORE_OPT_ADADELTA;
  const bool betas = kind == BORE_OPT_ADAM || kind == BORE_OPT_ADAMAX || kind == BORE_OPT_NADAM;
  BORE_CHECK(o.lr > 0.f, "%s: learning_rate must be > 0, got %g", who, o.lr);
  BORE_CHECK(!(rho || betas) || (o.b1 >= 0.f && o.b1 < 1.f), "%s: %s must be in [0, 1), got %g", who,
             rho ? "rho" : "beta_1", o.b1);
  BORE_CHECK(!betas || (o.b2 >= 0.f && o.b2 < 1.f), "%s: beta_2 must be in [0, 1), got %g", who, o.b2);
  // eps > 0 keeps the zero-gradient, zero-slot padding parameters of the kernels at exactly zero (0/0 else)
  BORE_CHECK(kind == BORE_OPT_ADAM ? o.eps >= 0.f : o.eps > 0.f, "%s: epsilon must be %s 0, got %g", who,
             kind == BORE_OPT_ADAM ? ">=" : ">", o.eps);
  BORE_CHECK(o.momentum >= 0.f && o.momentum < 1.f, "%s: momentum must be in [0, 1), got %g", who, o.momentum);
  BORE_CHECK(o.init_acc >= 0.f, "%s: initial_accumulator_value must be >= 0, got %g", who, o.init_acc);
  BORE_CHECK(hp[6] == 0.f || hp[6] == 1.f, "%s: centered must be 0 or 1, got %g", who, hp[6]);
  BORE_CHECK(!(kind == BORE_OPT_RMSPROP && o.centered && o.momentum > 0.f),
             "%s: RMSprop(centered=True, momentum>0) needs a third slot per parameter, which no kernel keeps", who);
  if (kind != BORE_OPT_RMSPROP) { o.momentum = 0.f; o.centered = 0; }
  if (kind != BORE_OPT_ADAGRAD) o.init_acc = 0.f;
  if (!rho && !betas) o.b1 = 0.f;
  if (!betas) o.b2 = 0.f;
  return 0;
}

int lr_schedule_from_array(int kind, const float *sp, int n_sp, LrSchedule &o, const char *who) {
  BORE_CHECK(kind >= BORE_LR_CONSTANT && kind <= BORE_LR_PIECEWISE,
             "%s: unknown schedule kind %d (BORE_LR_CONSTANT .. BORE_LR_PIECEWISE)", who, kind);
  static const int n_of[] = {0, 4, 4, 5};  // sp entries of the kinds before BORE_LR_PIECEWISE
  BORE_CHECK(n_sp >= 0 && (n_sp == 0 || sp != nullptr), "%s: %d schedule parameters, array NULL", who, n_sp);
  if (kind == BORE_LR_PIECEWISE)
    BORE_CHECK(n_sp % 2 == 1 && n_sp >= 3 && n_sp <= 2 * BORE_LR_MAX_BOUNDARIES + 1,
               "%s: PiecewiseConstantDecay takes n boundaries and n + 1 values, 1 <= n <= %d (got %d parameters)",
               who, BORE_LR_MAX_BOUNDARIES, n_sp);
  else
    BORE_CHECK(n_sp == n_of[kind], "%s: schedule kind %d takes %d parameters, got %d", who, kind, n_of[kind], n_sp);
  for (int i = 0; i < n_sp; ++i) BORE_CHECK(isfinite(sp[i]), "%s: schedule parameter %d is %g", who, i, (double)sp[i]);
  o = LrSchedule{};
  o.kind = kind;
  if (kind == BORE_LR_PIECEWISE) {
    o.n = n_sp / 2;
    for (int i = 0; i < o.n; ++i) {
      BORE_CHECK(i == 0 || sp[i] > sp[i - 1], "%s: boundaries must be strictly increasing (%g after %g)", who,
                 (double)sp[i], (double)sp[i - 1]);
      o.bound[i] = sp[i];
    }
    for (int i = 0; i <= o.n; ++i) o.value[i] = sp[o.n + i];
  } else if (kind != BORE_LR_CONSTANT) {
    o.initial = sp[0];
    o.decay_steps = sp[1];
    BORE_CHECK(o.decay_steps > 0.f, "%s: decay_steps must be > 0, got %g", who, (double)o.decay_steps);
    const float flag = sp[n_sp - 1];
    BORE_CHECK(flag == 0.f || flag == 1.f, "%s: %s must be 0 or 1, got %g", who,
               kind == BORE_LR_POLYNOMIAL ? "cycle" : "staircase", (double)flag);
    o.flag = flag != 0.f;
    if (kind == BORE_LR_POLYNOMIAL) { o.end = sp[2]; o.power = sp[3]; }
    else o.rate = sp[2];
  }
  return 0;
}

extern "C" {

int bore_abi_version(void) { return BORE_ABI_VERSION; }
const char *bore_last_error(void) { return g_err; }

int bore_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int bore_mlp_create(int n_layers, const int *dims, const int *acts, int n_models, int device,
                    bore_mlp **out) {
  BORE_CHECK(out != nullptr, "bore_mlp_create: out is NULL");
  BORE_CHECK(n_layers >= 1 && n_layers <= BORE_MAX_LAYERS,
             "bore_mlp_create: n_layers=%d outside [1,%d]", n_layers, BORE_MAX_LAYERS);
  BORE_CHECK(n_models >= 1, "bore_mlp_create: n_models=%d", n_models);
  BORE_CHECK(dims[0] >= 1 && dims[0] <= BORE_MAX_DIM, "bore_mlp_create: input dim %d outside [1,%d]",
             dims[0], BORE_MAX_DIM);
  BORE_CHECK(dims[n_layers] == 1,
             "bore_mlp_create: output dimension must be 1 (bore/base.py:19-21), got %d",
             dims[n_layers]);
  for (int l = 1; l < n_layers; ++l)
    BORE_CHECK(dims[l] >= 1 && dims[l] <= BORE_MAX_WIDTH,
               "bore_mlp_create: hidden width %d outside [1,%d]", dims[l], BORE_MAX_WIDTH);
  for (int l = 0; l < n_layers; ++l)
    BORE_CHECK(acts[l] >= BORE_ACT_LINEAR && acts[l] <= BORE_ACT_EXPONENTIAL,
               "bore_mlp_create: unknown activation code %d", acts[l]);
  MlpDesc d;
  memset(&d, 0, sizeof(d));
  d.n_layers = n_layers;
  int off = 0;
  for (int l = 0; l <= n_layers; ++l) d.dims[l] = dims[l];
  for (int l = 0; l < n_layers; ++l) {
    d.act[l] = acts[l];
    d.w_off[l] = off; off += dims[l] * dims[l + 1];
    d.b_off[l] = off; off += dims[l + 1];
  }
  d.n_params = off;
  // the limits above are necessary, not sufficient: a net inside them can still need more shared
  // memory than an SM has.  Refuse it here rather than at its first predict / fit / argmax.
  if (mlp_eval_check_envelope(d) != 0 || fit_check_envelope(d) != 0) return -1;
  BORE_CHECK(bore_device_count() > 0,
             "bore_mlp_create: no CUDA device visible -- bore_b200 has no CPU fallback");
  BORE_CUDA(cudaSetDevice(device));
  bore_mlp *h = new bore_mlp();
  memset(h, 0, sizeof(*h));
  h->pack = new MlpPackCache();
  memset(h->pack, 0, sizeof(*h->pack));
  h->desc = d;
  h->n_models = n_models;
  h->opt = OptHyper{1e-3f, 0.9f, 0.999f, 1e-7f, 0.f, 0.f, BORE_OPT_ADAM, 0};  // Keras "adam"
  h->device = device;
  cudaDeviceProp prop;
  BORE_CUDA(cudaGetDeviceProperties(&prop, device));
  h->sm_count = prop.multiProcessorCount;
  const size_t nb = (size_t)n_models * off * sizeof(float);
  BORE_CUDA(cudaMalloc(&h->params, nb));
  BORE_CUDA(cudaMalloc(&h->adam_m, nb));
  BORE_CUDA(cudaMalloc(&h->adam_v, nb));
  BORE_CUDA(cudaMalloc(&h->adam_t, n_models * sizeof(long long)));
  BORE_CUDA(cudaMalloc(&h->opt_cache, n_models * sizeof(float)));
  BORE_CUDA(cudaMemset(h->params, 0, nb));
  BORE_CHECK_RC(opt_reset_state(h->opt, h->adam_m, h->adam_v, off, h->adam_t, h->opt_cache, n_models, 0));
  BORE_CUDA(cudaDeviceSynchronize());
  *out = h;
  return 0;
}

int bore_mlp_destroy(bore_mlp *h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  cudaFree(h->params);
  cudaFree(h->adam_m);
  cudaFree(h->adam_v);
  cudaFree(h->adam_t);
  cudaFree(h->opt_cache);
  if (h->pack) {
    for (int v = 0; v < 4; ++v) cudaFree(h->pack->buf[v]);
    delete h->pack;
  }
  if (h->tab_done) {
    cudaEventSynchronize(h->tab_done);
    cudaEventDestroy(h->tab_done);
  }
  if (h->tab_pinned) cudaFreeHost(h->tab_pinned);
  delete h;
  return 0;
}

int bore_mlp_num_params(const bore_mlp *h) { return h ? h->desc.n_params : -1; }
int bore_mlp_num_models(const bore_mlp *h) { return h ? h->n_models : -1; }

#define CHECK_MODEL(h, model)                                                              \
  BORE_CHECK((h) != nullptr, "NULL handle");                                               \
  BORE_CHECK((model) >= 0 && (model) < (h)->n_models, "model index %d outside [0,%d)", model, \
             (h)->n_models);                                                               \
  BORE_CUDA(cudaSetDevice((h)->device))

int bore_mlp_set_weights(bore_mlp *h, int model, const float *params_host) {
  CHECK_MODEL(h, model);
  const size_t nb = (size_t)h->desc.n_params * sizeof(float);
  // fit / argmax run on the caller's streams, which a legacy-stream copy is not ordered against
  // when they are non-blocking: drain the device first (parameter I/O is rare)
  BORE_CUDA(cudaDeviceSynchronize());
  BORE_CUDA(cudaMemcpy(h->params + (size_t)model * h->desc.n_params, params_host, nb,
                       cudaMemcpyHostToDevice));
  return 0;
}

int bore_mlp_get_weights(bore_mlp *h, int model, float *params_host) {
  CHECK_MODEL(h, model);
  const size_t nb = (size_t)h->desc.n_params * sizeof(float);
  BORE_CUDA(cudaDeviceSynchronize());  // see bore_mlp_set_weights
  BORE_CUDA(cudaMemcpy(params_host, h->params + (size_t)model * h->desc.n_params, nb,
                       cudaMemcpyDeviceToHost));
  return 0;
}

int bore_mlp_set_adam_state(bore_mlp *h, int model, const float *m_host, const float *v_host,
                            int64_t iterations) {
  CHECK_MODEL(h, model);
  const size_t np = h->desc.n_params, nb = np * sizeof(float);
  BORE_CUDA(cudaDeviceSynchronize());
  BORE_CUDA(cudaMemcpy(h->adam_m + model * np, m_host, nb, cudaMemcpyHostToDevice));
  BORE_CUDA(cudaMemcpy(h->adam_v + model * np, v_host, nb, cudaMemcpyHostToDevice));
  long long t = iterations;
  BORE_CUDA(cudaMemcpy(h->adam_t + model, &t, sizeof(t), cudaMemcpyHostToDevice));
  return 0;
}

int bore_mlp_get_adam_state(bore_mlp *h, int model, float *m_host, float *v_host,
                            int64_t *iterations) {
  CHECK_MODEL(h, model);
  const size_t np = h->desc.n_params, nb = np * sizeof(float);
  BORE_CUDA(cudaDeviceSynchronize());
  BORE_CUDA(cudaMemcpy(m_host, h->adam_m + model * np, nb, cudaMemcpyDeviceToHost));
  BORE_CUDA(cudaMemcpy(v_host, h->adam_v + model * np, nb, cudaMemcpyDeviceToHost));
  long long t = 0;
  BORE_CUDA(cudaMemcpy(&t, h->adam_t + model, sizeof(t), cudaMemcpyDeviceToHost));
  *iterations = t;
  return 0;
}

int bore_mlp_reset_optimizer(bore_mlp *h, int model0, int count, void *stream) {
  BORE_CHECK(h != nullptr, "NULL handle");
  BORE_CHECK(model0 >= 0 && count >= 1 && model0 + count <= h->n_models,
             "bore_mlp_reset_optimizer: models [%d,%d) outside [0,%d)", model0, model0 + count,
             h->n_models);
  BORE_CUDA(cudaSetDevice(h->device));
  const size_t np = h->desc.n_params;
  return opt_reset_state(h->opt, h->adam_m + model0 * np, h->adam_v + model0 * np, np, h->adam_t + model0,
                         h->opt_cache + model0, count, (cudaStream_t)stream);
}

// a change of kind: every model starts from the new kind's initial state (Keras builds fresh slots)
static int mlp_change_optimizer(bore_mlp *h, const OptHyper &o) {
  if (o.kind != h->opt.kind) {
    BORE_CUDA(cudaSetDevice(h->device));
    BORE_CUDA(cudaDeviceSynchronize());
    BORE_CHECK_RC(opt_reset_state(o, h->adam_m, h->adam_v, h->desc.n_params, h->adam_t, h->opt_cache,
                                  h->n_models, 0));
    BORE_CUDA(cudaDeviceSynchronize());
  }
  h->opt = o;
  return 0;
}

int bore_mlp_set_optimizer(bore_mlp *h, float lr, float beta1, float beta2, float eps) {
  BORE_CHECK(h != nullptr, "NULL handle");
  BORE_CHECK(lr > 0.f && beta1 >= 0.f && beta1 < 1.f && beta2 >= 0.f && beta2 < 1.f && eps >= 0.f,
             "bore_mlp_set_optimizer: invalid Adam hyper-parameters");
  return mlp_change_optimizer(h, OptHyper{lr, beta1, beta2, eps, 0.f, 0.f, BORE_OPT_ADAM, 0});
}

int bore_mlp_set_optimizer_kind(bore_mlp *h, int kind, const float *hp) {
  OptHyper o;
  BORE_CHECK_RC(opt_from_array(kind, hp, o, "bore_mlp_set_optimizer_kind"));
  BORE_CHECK(h != nullptr, "NULL handle");
  return mlp_change_optimizer(h, o);
}

int bore_mlp_set_lr_schedule(bore_mlp *h, int kind, const float *sp, int n_sp) {
  LrSchedule s;
  BORE_CHECK_RC(lr_schedule_from_array(kind, sp, n_sp, s, "bore_mlp_set_lr_schedule"));
  BORE_CHECK(h != nullptr, "NULL handle");
  h->sched = s;  // the state is kept, as Keras keeps its slots under a new rate
  return 0;
}

int bore_mlp_get_nadam_cache(bore_mlp *h, int model, float *cache_host) {
  CHECK_MODEL(h, model);
  BORE_CHECK(cache_host != nullptr, "NULL argument");
  BORE_CUDA(cudaDeviceSynchronize());
  BORE_CUDA(cudaMemcpy(cache_host, h->opt_cache + model, sizeof(float), cudaMemcpyDeviceToHost));
  return 0;
}

int bore_mlp_set_nadam_cache(bore_mlp *h, int model, float cache) {
  CHECK_MODEL(h, model);
  BORE_CUDA(cudaDeviceSynchronize());
  BORE_CUDA(cudaMemcpy(h->opt_cache + model, &cache, sizeof(float), cudaMemcpyHostToDevice));
  return 0;
}

int bore_mlp_set_regularizers(bore_mlp *h, const float *l2_kernel_host, const float *l2_bias_host) {
  BORE_CHECK(h != nullptr && l2_kernel_host && l2_bias_host, "NULL argument");
  for (int l = 0; l < h->desc.n_layers; ++l) {
    BORE_CHECK(l2_kernel_host[l] >= 0.f && l2_bias_host[l] >= 0.f, "negative l2 factor");
    h->l2k[l] = l2_kernel_host[l];
    h->l2b[l] = l2_bias_host[l];
  }
  return 0;
}

int bore_mlp_set_l1_regularizers(bore_mlp *h, const float *l1_kernel_host, const float *l1_bias_host) {
  BORE_CHECK(h != nullptr && l1_kernel_host && l1_bias_host, "NULL argument");
  for (int l = 0; l < h->desc.n_layers; ++l)
    for (const float f : {l1_kernel_host[l], l1_bias_host[l]})
      BORE_CHECK(isfinite(f) && f >= 0.f, "l1 factor of layer %d is %g: it must be finite and >= 0", l, (double)f);
  for (int l = 0; l < h->desc.n_layers; ++l) {
    h->l1k[l] = l1_kernel_host[l];
    h->l1b[l] = l1_bias_host[l];
  }
  return 0;
}

int bore_mlp_set_dropout(bore_mlp *h, int n, const float *rates_host, const uint32_t *seeds_host) {
  BORE_CHECK(n >= 0 && n < BORE_MAX_LAYERS, "bore_mlp_set_dropout: %d hidden layers, outside [0, %d]", n,
             BORE_MAX_LAYERS - 1);
  BORE_CHECK(n == 0 || (rates_host != nullptr && seeds_host != nullptr), "bore_mlp_set_dropout: NULL argument");
  for (int l = 0; l < n; ++l)
    BORE_CHECK(isfinite(rates_host[l]) && rates_host[l] >= 0.f && rates_host[l] < 1.f,
               "bore_mlp_set_dropout: rate of hidden layer %d is %g: it must be finite and in [0, 1)", l,
               (double)rates_host[l]);
  BORE_CHECK(h != nullptr, "NULL handle");
  BORE_CHECK(n == h->desc.n_layers - 1, "bore_mlp_set_dropout: the net has %d hidden layers, got %d",
             h->desc.n_layers - 1, n);
  for (int l = 0; l < BORE_MAX_LAYERS; ++l) {  // the weights and the optimizer state are kept
    h->drop_rate[l] = l < n ? rates_host[l] : 0.f;
    h->drop_seed[l] = l < n ? seeds_host[l] : 0u;
  }
  return 0;
}

int bore_mlp_params_dev(bore_mlp *h, float **params_dev) {
  BORE_CHECK(h != nullptr && params_dev != nullptr, "NULL argument");
  *params_dev = h->params;
  return 0;
}

int bore_mlp_predict(bore_mlp *h, int model, const float *X_dev, int S, float *out_dev,
                     void *stream) {
  BORE_NVTX("bore:predict (K0)");
  CHECK_MODEL(h, model);
  BORE_CHECK(S >= 0, "bore_mlp_predict: S=%d", S);
  return launch_mlp_eval(h, model, false, BORE_TRANSFORM_IDENTITY, 0, X_dev, S, out_dev, nullptr,
                         nullptr, nullptr, (cudaStream_t)stream);
}

int bore_mlp_predict_multi(bore_mlp *h, int model0, int n_models, const float *X_dev,
                           int points_per_model, float *out_dev, void *stream) {
  BORE_CHECK(h != nullptr, "NULL handle");
  BORE_CHECK(model0 >= 0 && n_models >= 1 && model0 + n_models <= h->n_models,
             "bore_mlp_predict_multi: models [%d,%d) outside [0,%d)", model0, model0 + n_models,
             h->n_models);
  BORE_CHECK(points_per_model >= 1 && X_dev && out_dev, "bore_mlp_predict_multi: bad arguments");
  BORE_CUDA(cudaSetDevice(h->device));
  return launch_mlp_eval_multi(h, model0, n_models, points_per_model, false, BORE_TRANSFORM_IDENTITY, 0,
                               X_dev, out_dev, nullptr, nullptr, (cudaStream_t)stream);
}

int bore_mlp_value_and_grad(bore_mlp *h, int model, int transform, int negate, const float *X_dev,
                            int S, float *f_dev, float *g_dev, void *stream) {
  BORE_NVTX("bore:value_and_grad (K2)");
  CHECK_MODEL(h, model);
  BORE_CHECK(S >= 0, "bore_mlp_value_and_grad: S=%d", S);
  BORE_CHECK(transform >= 0 && transform <= BORE_TRANSFORM_EXP, "unknown transform code %d",
             transform);
  return launch_mlp_eval(h, model, true, transform, negate, X_dev, S, f_dev, g_dev, nullptr,
                         nullptr, (cudaStream_t)stream);
}

}  // extern "C"

// ---------------------------------------------------------------- FFMA peak microbenchmark
namespace {
__global__ void __launch_bounds__(512) ffma_peak_kernel(float *out, int iters, float a, float b) {
  float acc[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) acc[i] = (float)(threadIdx.x + i);
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int r = 0; r < 8; ++r)
#pragma unroll
      for (int i = 0; i < 16; ++i) acc[i] = fmaf(acc[i], a, b);
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 16; ++i) s += acc[i];
  if (s == 123.456f) out[0] = s;  // keep the chain alive
}
}  // namespace

extern "C" int bore_bench_ffma_peak(int device, int iters, double *tflops_out) {
  BORE_CHECK(tflops_out != nullptr, "NULL argument");
  BORE_CHECK(bore_device_count() > 0, "no CUDA device visible");
  BORE_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  BORE_CUDA(cudaGetDeviceProperties(&prop, device));
  float *out;
  BORE_CUDA(cudaMalloc(&out, 4));
  const int threads = 512, grid = prop.multiProcessorCount * 4;
  if (iters <= 0) iters = 4096;
  cudaEvent_t e0, e1;
  BORE_CUDA(cudaEventCreate(&e0));
  BORE_CUDA(cudaEventCreate(&e1));
  double best = 0;
  for (int rep = 0; rep < 5; ++rep) {
    BORE_CUDA(cudaEventRecord(e0));
    ffma_peak_kernel<<<grid, threads>>>(out, iters, 0.999f, 0.001f);
    BORE_CUDA(cudaEventRecord(e1));
    BORE_CUDA(cudaEventSynchronize(e1));
    float ms = 0;
    BORE_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    const double flop = 2.0 * 16 * 8 * (double)iters * threads * (double)grid;
    const double tf = flop / (ms * 1e-3) / 1e12;
    if (rep > 0 && tf > best) best = tf;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(out);
  *tflops_out = best;
  return 0;
}
