/*
 * bore_b200.h -- C ABI of libbore_b200.so: the B200-native (sm_100a) replacement for the
 * third-party numerics underneath ltiao/bore's BORE-MLP hot path.
 *
 * The reference (pure Python, /root/reference) has no FFI of its own; everything below
 * replaces a *library call site* in it.  Each entry point cites the reference call it
 * stands in for.  The only caller is the Python host layer `bore_b200/_lib.py` (ctypes).
 *
 * Conventions
 *   - every function returns 0 on success, <0 on error; bore_last_error() gives the text
 *     (thread-local).
 *   - `*_dev` pointers are device pointers owned by the caller (e.g. torch `data_ptr()`);
 *     `*_host` pointers are host pointers.  No torch types cross this boundary.
 *   - `stream` is a `cudaStream_t` passed as void* (NULL = legacy default stream).
 *     Kernels are enqueued on it; functions do not synchronise unless documented.
 *   - handles are not thread-affine: every call sets the CUDA device of its handle
 *     (HpBandSter calls get_config / new_result from different threads,
 *     bore/plugins/hpbandster/base.py:216,276).
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef BORE_B200_H
#define BORE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BORE_ABI_VERSION 1

/* activations of a Dense layer or an LSTM cell (Keras names: linear, relu, elu, sigmoid, tanh, selu,
 * softplus, softsign, hard_sigmoid, exponential) */
enum { BORE_ACT_LINEAR = 0, BORE_ACT_RELU = 1, BORE_ACT_ELU = 2, BORE_ACT_SIGMOID = 3,
       BORE_ACT_TANH = 4, BORE_ACT_SELU = 5, BORE_ACT_SOFTPLUS = 6, BORE_ACT_SOFTSIGN = 7,
       BORE_ACT_HARD_SIGMOID = 8, BORE_ACT_EXPONENTIAL = 9 };
/* output transforms, TRANSFORMS of bore/plugins/hpbandster/base.py:18 */
enum { BORE_TRANSFORM_IDENTITY = 0, BORE_TRANSFORM_SIGMOID = 1, BORE_TRANSFORM_EXP = 2 };
/* optimizers of the training kernels (Keras names: adam, rmsprop, adagrad, adadelta, adamax, nadam);
 * bore_mlp_set_optimizer_kind / bore_lstm_set_optimizer_kind take BORE_OPT_NHP hyper-parameters */
enum { BORE_OPT_ADAM = 0, BORE_OPT_RMSPROP = 1, BORE_OPT_ADAGRAD = 2, BORE_OPT_ADADELTA = 3,
       BORE_OPT_ADAMAX = 4, BORE_OPT_NADAM = 5 };
#define BORE_OPT_NHP 7
/* learning-rate schedules of the training kernels (keras.optimizers.schedules: ExponentialDecay,
 * InverseTimeDecay, PolynomialDecay, PiecewiseConstantDecay); bore_mlp_set_lr_schedule /
 * bore_lstm_set_lr_schedule.  BORE_LR_CONSTANT: the optimizer's learning_rate at every step. */
enum { BORE_LR_CONSTANT = 0, BORE_LR_EXPONENTIAL = 1, BORE_LR_INVERSE_TIME = 2, BORE_LR_POLYNOMIAL = 3,
       BORE_LR_PIECEWISE = 4 };
#define BORE_LR_MAX_BOUNDARIES 16
/* per-start termination status, scipy.optimize.OptimizeResult.status for L-BFGS-B */
enum { BORE_STATUS_CONVERGED = 0, BORE_STATUS_LIMIT = 1, BORE_STATUS_ABNORMAL = 2 };

/* Necessary bounds of a net, not sufficient ones: the kernels keep a model's weights in one SM's
 * shared memory, so wide and deep nets with a large input dimension can exceed it inside these
 * limits.  bore_mlp_create refuses such a net and names the shared memory it would need (DESIGN.md,
 * "The net-shape envelope"). */
#define BORE_MAX_LAYERS 8     /* Dense layers per model, final layer included */
#define BORE_MAX_WIDTH 128    /* widest hidden layer */
#define BORE_MAX_DIM 512      /* input dimension */
#define BORE_LBFGSB_MAXCOR 10 /* upper limit of the `m` (maxcor) option */

typedef struct bore_mlp bore_mlp; /* opaque: M independent MLPs of one architecture */

int bore_abi_version(void);
const char *bore_last_error(void);
/* number of visible CUDA devices (0 => every compute call will fail) */
int bore_device_count(void);

/* ---- model container ---------------------------------------------------------------
 * Replaces keras.Sequential + Dense as built at README.rst:60-64, bore/models.py:9-21.
 * dims[0..n_layers] = input dim, hidden widths..., output dim (must be 1);
 * acts[0..n_layers-1] = BORE_ACT_*.  n_models independent weight sets (seeds / BO
 * problems / per-budget classifiers) share the architecture.  Parameters are fp32 in
 * Keras get_weights() order: [W0 (in,out) row-major, b0, W1, b1, ...], flat.           */
int bore_mlp_create(int n_layers, const int *dims, const int *acts, int n_models,
                    int device, bore_mlp **out);
int bore_mlp_destroy(bore_mlp *h);
int bore_mlp_num_params(const bore_mlp *h);
int bore_mlp_num_models(const bore_mlp *h);
/* keras Model.set_weights / get_weights (host buffers, n_params floats); synchronous */
int bore_mlp_set_weights(bore_mlp *h, int model, const float *params_host);
int bore_mlp_get_weights(bore_mlp *h, int model, float *params_host);
/* Adam slots m, v (n_params floats each) -- slot 0 and slot 1 of the other kinds -- and the step
 * counter `iterations`; Keras keeps them alive across fit() calls on one model (README.rst:93
 * loop).  synchronous                                                                   */
int bore_mlp_set_adam_state(bore_mlp *h, int model, const float *m_host,
                            const float *v_host, int64_t iterations);
int bore_mlp_get_adam_state(bore_mlp *h, int model, float *m_host, float *v_host,
                            int64_t *iterations);
/* reset the optimizer state of models [model0, model0+count) on `stream` (what re-compiling a
 * Keras model does to its optimizer): zero slots and `iterations` -- Adagrad's accumulator at
 * initial_accumulator_value, Nadam's momentum cache at 1; asynchronous                     */
int bore_mlp_reset_optimizer(bore_mlp *h, int model0, int count, void *stream);
/* Adam hyper-parameters (keras.optimizers.Adam(learning_rate, beta_1, beta_2, epsilon));
 * defaults are Keras' "adam": 1e-3, 0.9, 0.999, 1e-7.  Makes Adam the handle's optimizer; coming
 * from another kind, every model's state is reset as bore_mlp_set_optimizer_kind does.     */
int bore_mlp_set_optimizer(bore_mlp *h, float lr, float beta1, float beta2, float eps);
/* The handle's optimizer: kind = BORE_OPT_*, hp[BORE_OPT_NHP] =
 *   {learning_rate, beta_1 or rho, beta_2, epsilon, momentum, initial_accumulator_value, centered}
 * with the Keras 2.5 meaning of each (entries a kind does not have are ignored):
 *   Adam, Adamax, Nadam  learning_rate, beta_1, beta_2 in [0,1), epsilon
 *   RMSprop              learning_rate, rho in [0,1), epsilon, momentum in [0,1), centered (0 / 1);
 *                        centered with momentum > 0 is refused (a third slot per parameter)
 *   Adagrad              learning_rate, epsilon, initial_accumulator_value >= 0
 *   Adadelta             learning_rate, rho in [0,1), epsilon
 * learning_rate > 0; epsilon > 0 (Adam: >= 0).  Unknown kinds are refused.  A new kind resets every
 * model's state to that kind's initial values: zero slots and `iterations`, Adagrad's accumulator
 * (slot 0) at initial_accumulator_value, Nadam's momentum cache at 1.  The same kind only changes the
 * hyper-parameters.  bore_mlp_{get,set}_adam_state read and write slot 0 and slot 1 of any kind
 * (DESIGN.md, "Optimizers", has the slot of each kind).  Synchronous.                         */
int bore_mlp_set_optimizer_kind(bore_mlp *h, int kind, const float *hp);
/* The handle's learning-rate schedule: kind = BORE_LR_*, sp[n_sp] =
 *   BORE_LR_CONSTANT      nothing (n_sp = 0, sp may be NULL): learning_rate of the optimizer, the state at create
 *   BORE_LR_EXPONENTIAL   {initial_learning_rate, decay_steps, decay_rate, staircase (0 / 1)}
 *   BORE_LR_INVERSE_TIME  {initial_learning_rate, decay_steps, decay_rate, staircase (0 / 1)}
 *   BORE_LR_POLYNOMIAL    {initial_learning_rate, decay_steps, end_learning_rate, power, cycle (0 / 1)}
 *   BORE_LR_PIECEWISE     {boundaries b_0 < .. < b_{n-1}, values v_0 .. v_n}: n_sp = 2 n + 1, 1 <= n <=
 *                         BORE_LR_MAX_BOUNDARIES
 * with the Keras 2.5 meaning; every value finite and decay_steps > 0, else refused.  Update number t (1-based)
 * of a model uses the schedule at step t - 1, in fp32, as Keras' _decayed_lr evaluates it at `iterations`
 * before the increment, so a later fit continues the schedule.  The optimizer state is kept.  Nadam takes
 * no schedule (Keras 2.5 refuses one) and keeps its learning_rate.  Synchronous, host only.          */
int bore_mlp_set_lr_schedule(bore_mlp *h, int kind, const float *sp, int n_sp);
/* Nadam's momentum cache (Keras' m_cache, one fp32 scalar per model; 1 after a reset).  synchronous */
int bore_mlp_get_nadam_cache(bore_mlp *h, int model, float *cache_host);
int bore_mlp_set_nadam_cache(bore_mlp *h, int model, float cache);
/* l2 regularisers (keras.regularizers.l2) per Dense layer: l2_kernel[l] * sum(W_l^2) +
 * l2_bias[l] * sum(b_l^2) is added to the training loss (n_layers floats each; zeros = none).
 * The plugin regularises its hidden layers only (plugins/hpbandster/base.py:113-116,152-155). */
int bore_mlp_set_regularizers(bore_mlp *h, const float *l2_kernel_host, const float *l2_bias_host);
/* l1 regularisers (keras.regularizers.l1, the l1 half of l1_l2) per Dense layer: l1_kernel[l] * sum|W_l| +
 * l1_bias[l] * sum|b_l| is added to the training loss and to evaluate's, next to the l2 terms; the gradient
 * term is l1 * sign(w) with sign(0) = 0, as TF's Abs gradient.  n_layers floats each, finite and >= 0
 * (anything else is refused); zeros = none, the state at create.                                      */
int bore_mlp_set_l1_regularizers(bore_mlp *h, const float *l1_kernel_host, const float *l1_bias_host);
/* Dropout (keras.layers.Dropout) after each hidden layer, in training only: rates[l] and seeds[l] for the
 * output of Dense layer l, l < n = n_layers - 1 hidden layers; rate 0 is no dropout, every rate finite and
 * in [0, 1), else refused.  Arrays may be NULL when n = 0.  The mask of hidden layer l, unit j, minibatch
 * position i, model m at the step whose Keras `iterations` is t before its increment is Philox4x32-10 with
 * counter (t mod 2^32, t div 2^32, i, 65536 l + j div 4) and key (seeds[l], m): unit j is kept when output
 * word j mod 4 gives (w >> 8) 2^-24 >= rates[l], and scaled by fp32(1 / (1 - rates[l])) (DESIGN.md,
 * "Dropout").  evaluate, predict, value-and-gradient and the argmax see no dropout.  All rates are 0 at
 * create; setting dropout keeps the weights and the optimizer state.  Synchronous, host only.           */
int bore_mlp_set_dropout(bore_mlp *h, int n, const float *rates_host, const uint32_t *seeds_host);
/* device pointer of the flat parameter block [n_models][n_params] (for NCCL broadcast) */
int bore_mlp_params_dev(bore_mlp *h, float **params_dev);

/* ---- K0: batched forward -------------------------------------------------------------
 * Replaces keras Model.predict at bore/mixins.py:50.  X_dev [S][D] fp32 row-major,
 * out_dev [S] fp32 (model output, final activation applied).                            */
int bore_mlp_predict(bore_mlp *h, int model, const float *X_dev, int S, float *out_dev,
                     void *stream);

/* ---- K2: fused value + input-gradient --------------------------------------------------
 * Replaces the tf.function/GradientTape closure built by convert()
 * (bore/base.py:35-42, bore/decorators.py:48-65): f = T(sign*u(x)), g = df/dx with
 * sign = -1 when negate!=0 (the `_func_min` of bore/mixins.py:20), +1 otherwise
 * (`_func_max`, bore/mixins.py:97).  X_dev [S][D], f_dev [S], g_dev [S][D], all fp32.   */
int bore_mlp_value_and_grad(bore_mlp *h, int model, int transform, int negate,
                            const float *X_dev, int S, float *f_dev, float *g_dev,
                            void *stream);

/* ---- K1: fused training ----------------------------------------------------------------
 * Replaces keras Model.fit(X, z, epochs, batch_size, shuffle=True) compiled with the handle's optimizer
 * (Adam unless bore_mlp_set_optimizer_kind chose another) +
 * binary cross-entropy (README.rst:66,93; bore/plugins/hpbandster/base.py:156-157,184):
 * the whole run is one launch, one CTA group per model.  Models [model0, model0+count)
 * train concurrently, model j on rows [j*N, (j+1)*N) of X_dev/z_dev when
 * `shared_data == 0`, or all on the same N rows when `shared_data != 0`.
 *   X_dev [*][D] fp32, z_dev [*] fp32 (0/1 labels)
 *   perm_dev [count or 1][epochs][N] int32: the per-epoch shuffles (Keras draws them
 *     internally; made explicit so trajectories can be compared).  One set per model, or
 *     one shared set when `shared_perm != 0`.
 *   loss_out_dev [count][epochs] fp32: Keras' history["loss"] (sample-weighted running
 *     mean of the per-batch losses, each taken before its update); may be NULL.
 * Weights and Adam state of the handle are updated in place.                            */
int bore_mlp_fit(bore_mlp *h, int model0, int count, const float *X_dev,
                 const float *z_dev, int N, int shared_data, int batch_size, int epochs,
                 const int32_t *perm_dev, int shared_perm, float *loss_out_dev, void *stream);

/* How bore_mlp_fit maps models onto the GPU: 0 = automatic (default), 1 = one CTA per model
 * (throughput mode, many concurrent models), 2 = one 8-CTA thread-block cluster per model
 * (latency mode: the minibatch is split over 8 SMs, gradients meet in distributed shared
 * memory), 3 = tensor pipe (one CTA per model, every GEMM of a step as 3xTF32 mma.sync; hidden
 * widths <= 128, batch <= 64, 1-unit output layer, else an error) -- kept as the measured
 * answer to "would tensor cores help": slower than 1 and 2 on B200 (DESIGN.md, K1t), so never
 * picked automatically (BORE_FIT_MMA=1 in the environment prefers it), 4 = one 8-CTA cluster per
 * model with the hidden UNITS split over the CTAs (every CTA owns a column and a row slice of each
 * weight matrix, only activations and deltas cross SMs; needs a hidden layer, batch <= 64, else
 * an error).  Automatic picks 4 (else 2) while 8 * count <= number of SMs; BORE_FIT_UNIT=0 in the
 * environment skips 4.  Same results up to fp32 summation order.                             */
int bore_mlp_set_fit_mode(bore_mlp *h, int mode);

/* Keras Model.evaluate -> mean loss and `accuracy` (plugins/hpbandster/base.py:186).
 * out_host[0]=loss, out_host[1]=accuracy.  synchronous.                                 */
int bore_mlp_evaluate(bore_mlp *h, int model, const float *X_dev, const float *z_dev,
                      int N, float *out_host, void *stream);

/* ---- K1, weighted: Keras fit(..., sample_weight=w, class_weight={0: cw0, 1: cw1}) ------------
 * bore_mlp_fit with a loss weight per sample: sample i of a minibatch of nb weighs
 * w_i * cw[z_i] (w_i = 1 when w_dev is NULL; z_i is its 0/1 label, so the class weights also
 * apply to labels made on the device), and the minibatch loss is sum_i w_i cw[z_i] bce_i / nb
 * (+ the l2 terms): Keras' SUM_OVER_BATCH_SIZE, divided by the sample count, not by the weights.
 * history["loss"] keeps its form (the epoch mean weighs each minibatch by its sample count).
 *   w_dev: the layout of z_dev, [count][N] or one shared [N] when `shared_data != 0`; any
 *     values (zeros and negatives pass through, as in Keras).
 * Same kernels, fit modes, environment overrides and refusals as bore_mlp_fit.  With w_dev NULL
 * and class weights (1, 1) it is bore_mlp_fit; an all-ones w_dev gives the same bits too.    */
int bore_mlp_fit_weighted(bore_mlp *h, int model0, int count, const float *X_dev,
                          const float *z_dev, const float *w_dev, int N, int shared_data,
                          float class_weight0, float class_weight1, int batch_size, int epochs,
                          const int32_t *perm_dev, int shared_perm, float *loss_out_dev,
                          void *stream);

/* Keras evaluate(..., sample_weight=w) with class weights as in bore_mlp_fit_weighted:
 * out_host[0] = sum_i w_i cw[z_i] bce_i / N (+ l2), out_host[1] = sum_i w_i cw[z_i] [correct_i] /
 * sum_i w_i cw[z_i], 0 when the weights sum to 0.  w_dev [N] may be NULL.  synchronous.     */
int bore_mlp_evaluate_weighted(bore_mlp *h, int model, const float *X_dev, const float *z_dev,
                               const float *w_dev, float class_weight0, float class_weight1,
                               int N, float *out_host, void *stream);

/* ---- K1, ragged: problems with their own observation counts and epochs -----------------------
 * bore_mlp_fit_weighted for `count` problems that each hold N_p >= 1 observations and train for
 * epochs_p >= 0 epochs (n_host[p], epochs_host[p]; host arrays).  Problem p is model model0 + p and
 * computes what a fit of that model alone on its own data computes: minibatches of min(batch, N_p),
 * ceil(N_p / batch) steps per epoch (the last one short), Adam's `iterations` advanced by
 * epochs_p * ceil(N_p / batch), history["loss"] over its N_p samples.  epochs_p = 0 leaves the model
 * untouched (weights, Adam m / v and iterations).  With R, Q, E the prefix sums over the problems in
 * their order (64-bit: R_p = sum_{q<p} N_q, Q_p = sum_{q<p} epochs_q * N_q, E_p = sum_{q<p} epochs_q):
 *   X_dev [R_count][D], z_dev / w_dev [R_count]: problem p's rows are [R_p, R_p + N_p); w_dev may be NULL
 *   perm_dev: problem p's shuffles are the [epochs_p][N_p] int32 block at Q_p (indices in [0, N_p))
 *   loss_out_dev (may be NULL): problem p's epoch losses are the epochs_p floats at E_p
 * The batch size, the net and the class weights are shared.  Same kernels, fit modes, environment
 * overrides and refusals as bore_mlp_fit; the plans are made for the batch min(batch, max N_p) over the
 * problems that train, and the kernel is chosen for their number.  w_dev NULL with class weights (1, 1)
 * runs the unweighted arithmetic.  With every N_p = N and epochs_p = E this is bore_mlp_fit(_weighted)
 * with shared_data = shared_perm = 0, bit for bit.  The problems are launched longest first
 * (epochs_p * ceil(N_p / batch)); the results do not depend on the order.  Every argument is checked
 * before anything is enqueued.                                                                     */
int bore_mlp_fit_ragged(bore_mlp *h, int model0, int count, const float *X_dev, const float *z_dev,
                        const float *w_dev, const int32_t *n_host, const int32_t *epochs_host,
                        float class_weight0, float class_weight1, int batch_size, const int32_t *perm_dev,
                        float *loss_out_dev, void *stream);

/* ---- K3: batched bound-constrained L-BFGS-B -------------------------------------------
 * Replaces the per-start scipy.optimize.minimize(fun, x0, method="L-BFGS-B", jac=True,
 * bounds=..., options=dict(maxiter, ftol)) loop of bore/mixins.py:57-61 (also
 * bore/optimizers/base.py:56-60), with K2 as the objective.  All S starts advance on
 * device; the host only polls a counter.
 *   X0_dev [S][D] fp64 start points (clipped into the box like SciPy does)
 *   lo_host/hi_host [D] fp64 (+-inf allowed = unbounded side)
 *   m (maxcor, <= BORE_LBFGSB_MAXCOR), ftol, gtol, maxiter, maxfun, maxls: SciPy options
 *   work_dev: scratch of bore_lbfgsb_workspace_bytes(S, D, m) bytes
 * Outputs (device): x_dev [S][D] fp64, fun_dev [S] fp64, nit/nfev/status/task_dev [S]
 * int32 (task = SciPy's numeric task message code, e.g. 401/402/504; may be NULL).
 * Returns after all starts terminated (synchronises `stream`).  *rounds_out (may be
 * NULL) receives the number of lock-step evaluation rounds, *evals_out the total number
 * of K2 point evaluations performed.                                                    */
size_t bore_lbfgsb_workspace_bytes(int S, int D, int m);
/* Scratch bore_lbfgsb_minimize / _minimize_multi need for S starts on model handle `h`: a few
 * hundred bytes when the fused persistent kernel runs the call (weights and >= 2 starts fit in
 * one SM's shared memory -- every BASELINE.json config), else bore_lbfgsb_workspace_bytes.   */
size_t bore_lbfgsb_minimize_workspace_bytes(const bore_mlp *h, int S, int m);
/* How bore_lbfgsb_minimize / _minimize_multi run (process-wide): 0 = default rule -- ONE fused
 * persistent launch (a warp keeps its start in shared memory and evaluates the MLP itself) when
 * the model fits and S <= 4,096 (16,384 for problems of at most 16 dimensions), lock-step rounds of K2 + stepper launches above; 1 = always
 * rounds (the path bore_lbfgsb_step exposes); 2 = always fused when the model fits.
 * BORE_LB_FUSED=0 / 1 / 2 in the environment selects 1 / 0 / 2 at start-up.  Query workspace
 * sizes after changing it.                                                                  */
int bore_lbfgsb_set_mode(int mode);
int bore_lbfgsb_minimize(bore_mlp *h, int model, int transform, const double *X0_dev,
                         int S, const double *lo_host, const double *hi_host, int m,
                         double ftol, double gtol, int maxiter, int maxfun, int maxls,
                         void *work_dev, size_t work_bytes, double *x_dev,
                         double *fun_dev, int32_t *nit_dev, int32_t *nfev_dev,
                         int32_t *status_dev, int32_t *task_dev, int *rounds_out,
                         long long *evals_out, void *stream);

/* Measurement hooks for bench.py: when enabled, bore_lbfgsb_minimize brackets every kernel it
 * launches with CUDA events on `stream`; bore_lbfgsb_last_profile returns, for the last such
 * call, out[0] = K2 total ms, out[1] = stepper (or fused kernel) total ms, out[2] = rounds
 * (= launches of each kernel), out[3] = algorithmic bytes (DESIGN.md), out[4] = point
 * evaluations, out[5] = 1 when the fused persistent kernel ran, out[6] / out[7] = its grid /
 * block size.                                                                              */
int bore_lbfgsb_profile(int enable);
int bore_lbfgsb_last_profile(double *out8);

/* L-BFGS-B stepper alone, objective supplied by the caller (reverse communication):
 * used to pin the on-device algorithm against SciPy's setulb request by request, and by
 * minimize_multi_start() for objectives that are not a bore_mlp.
 *   bore_lbfgsb_init: set up S states from X0; first requests are written to xreq_dev
 *   bore_lbfgsb_step: consume f_dev[S] (fp32 or fp64 per `f_is_f64`), g_dev[S][D] for the
 *     starts that were pending, advance each to its next request or to termination.
 *     *pending_out = number of starts still asking for an evaluation (synchronises).
 *   xreq_dev [S][D] fp64: current trial point of every start; pend_dev [S] int32 flags. */
int bore_lbfgsb_init(const double *X0_dev, int S, int D, const double *lo_host,
                     const double *hi_host, int m, double ftol, double gtol, int maxiter,
                     int maxfun, int maxls, void *work_dev, size_t work_bytes,
                     double *xreq_dev, int32_t *pend_dev, int device, void *stream);
int bore_lbfgsb_step(const void *f_dev, const void *g_dev, int fg_is_f64, int S, int D,
                     void *work_dev, double *xreq_dev, int32_t *pend_dev,
                     int *pending_out, int device, void *stream);
int bore_lbfgsb_results(int S, int D, void *work_dev, double *x_dev, double *fun_dev,
                        int32_t *nit_dev, int32_t *nfev_dev, int32_t *status_dev,
                        int32_t *task_dev, int device, void *stream);

/* ---- K4: selection ---------------------------------------------------------------------
 * bore_topk_smallest replaces np.argpartition(f_init, kth=num_starts-1)
 * (bore/mixins.py:56): indices of the k smallest of f_dev[S] (ascending, ties by lower
 * index) into idx_dev[k].  With negate != 0 the ranking is on -f_dev (the reference ranks
 * f_init = -predict(X_init), bore/mixins.py:52).
 * bore_select_best replaces the final scan of bore/mixins.py:80-87: among starts with
 * status in {0,1} and keep_dev[i]!=0 (keep_dev may be NULL), the FIRST minimum of fun.
 * key_dev receives one int64: (orderable(-fun) << 31) | (0x7fffffff - (idx + idx_offset)),
 * or 0 if no start qualifies -- ready for one NCCL max all-reduce across ranks.         */
int bore_topk_smallest(const float *f_dev, int S, int k, int negate, int32_t *idx_dev,
                       void *work_dev, size_t work_bytes, int device, void *stream);
size_t bore_topk_workspace_bytes(int S, int k);
int bore_select_best(const double *fun_dev, const int32_t *status_dev,
                     const uint8_t *keep_dev, int S, int64_t idx_offset, int64_t *key_dev,
                     int device, void *stream);

/* ---- batched problems -----------------------------------------------------------------
 * BASELINE.json configs[3]: M independent BO problems (seeds / concurrent optimisations /
 * per-budget classifiers), each the reference's own `fit` + `argmax` (README.rst:93-96), advanced
 * together.  Training already takes a model range (bore_mlp_fit).  For the argmax, model
 * model0+b owns points / starts [b*per_model, (b+1)*per_model) of every array below; one CTA
 * per model evaluates its points, the L-BFGS-B stepper is the same kernel as for one model.
 *   bore_mlp_predict_multi       keras predict per problem (bore/mixins.py:50)
 *   bore_topk_smallest_groups    np.argpartition per problem (bore/mixins.py:56): idx_dev
 *                                [n_groups][k], indices WITHIN the group, ascending value
 *   bore_lbfgsb_minimize_multi   the scipy loop of bore/mixins.py:57-61 for every problem;
 *                                arguments as bore_lbfgsb_minimize with S = n_models *
 *                                starts_per_model
 *   bore_select_best_groups      the scan of bore/mixins.py:80-87 per problem: keys_dev
 *                                [n_groups] int64, low 31 bits = 0x7fffffff - index within the
 *                                group, 0 when no start of the group qualifies; keep_dev
 *                                (may be NULL) [n_groups][per_group] is the filter_fn mask     */
int bore_mlp_predict_multi(bore_mlp *h, int model0, int n_models, const float *X_dev,
                           int points_per_model, float *out_dev, void *stream);
int bore_topk_smallest_groups(const float *f_dev, int n_groups, int per_group, int k, int negate,
                              int32_t *idx_dev, int device, void *stream);
int bore_lbfgsb_minimize_multi(bore_mlp *h, int model0, int n_models, int starts_per_model,
                               int transform, const double *X0_dev, const double *lo_host,
                               const double *hi_host, int m, double ftol, double gtol, int maxiter,
                               int maxfun, int maxls, void *work_dev, size_t work_bytes,
                               double *x_dev, double *fun_dev, int32_t *nit_dev, int32_t *nfev_dev,
                               int32_t *status_dev, int32_t *task_dev, int *rounds_out,
                               long long *evals_out, void *stream);
int bore_select_best_groups(const double *fun_dev, const int32_t *status_dev,
                            const uint8_t *keep_dev, int n_groups, int per_group, int64_t *keys_dev,
                            int device, void *stream);

/* ---- C1: the one collective of the sharded argmax ---------------------------------------
 * Every rank holds the same weights and its own shard of the start points (the loop of
 * bore/mixins.py:57-61 split over the GPUs); bore_select_best(..., idx_offset = first global
 * index of the shard) gives its packed key, and ONE max all-reduce agrees on the winner:
 * ncclAllReduce(ncclMax, ncclInt64, count 1) on `nccl_comm` (an ncclComm_t), in place, on
 * `stream`.  The winner's global index is 0x7fffffff - (key & 0x7fffffff); key 0 = no start
 * qualified on any rank.  NCCL is looked up in the process at call time (no link dependency). */
int bore_allreduce_maxloc(void *nccl_comm, int64_t *key_dev, void *stream);

/* ---- data step either side of the path (SURVEY.md section 8f, row 2) --------------------
 * bore_quantile_labels replaces Record.load_classification_data (bore/data.py:31-35) for
 * n_problems target vectors y_dev [n_problems][N] (fp64) at once: tau = np.quantile(y, q)
 * (method "linear": virtual index (N-1)*q, numpy's _lerp between the two neighbouring order
 * statistics; NaN if the problem holds a NaN) and z = np.less(y, tau), STRICT.  Outputs (each
 * may be NULL): z_f32_dev [n_problems][N] as 0.f/1.f (what bore_mlp_fit consumes), z_u8_dev the
 * same as bytes, tau_dev [n_problems].  Bit-identical to numpy; N <= 16384 (one CTA sorts a
 * problem's targets in shared memory).
 * bore_is_duplicate replaces Record.is_duplicate (bore/data.py:42-48), the body of the
 * plugin's filter_fn (bore/plugins/hpbandster/base.py:227-231): candidate c of group g
 * (x_dev [n_groups][per_group][D]) is a duplicate if np.allclose(x_prev, x, rtol, atol) holds for
 * any of the group's stored rows x_prev_dev [n_groups][n_prev][D], i.e. for every coordinate
 * |x_prev - x| <= atol + rtol*|x| (x finite) or x_prev == x.  dup_dev / keep_dev (each may be
 * NULL) receive the flag / its negation per candidate; keep_dev is the mask bore_select_best
 * and bore_select_best_groups take.                                                       */
/* bore_truncnorm_distort replaces maybe_distort / truncated_normal (bore/base.py:45-64) for
 * n_points suggestions at once: out = truncnorm(a, b, loc, scale).rvs with a = (lo - loc)/scale,
 * b = (hi - loc)/scale per coordinate.  u_dev [n_points][D] holds the uniform variates scipy's
 * rvs would draw from the caller's random_state (one per coordinate, in order: draw them on the
 * host with random_state.uniform(size=(n_points, D)) to keep the stream), lo_dev / hi_dev [D].
 * Within 1e-9 of scipy (fp64 normcdf / normcdfinv instead of scipy's log-space ppf).       */
int bore_truncnorm_distort(const double *loc_dev, int n_points, int D, double scale,
                           const double *lo_dev, const double *hi_dev, const double *u_dev,
                           double *out_dev, int device, void *stream);
int bore_quantile_labels(const double *y_dev, int n_problems, int N, double q, float *z_f32_dev,
                         uint8_t *z_u8_dev, double *tau_dev, int device, void *stream);
int bore_is_duplicate(const double *x_dev, int n_groups, int per_group, const double *x_prev_dev,
                      int n_prev, int D, double rtol, double atol, uint8_t *dup_dev,
                      uint8_t *keep_dev, int device, void *stream);
/* Ragged forms of the two above.  bore_quantile_labels_ragged: problem p holds n_host[p] >= 1 targets
 * (<= 16384), y_dev / z_f32_dev / z_u8_dev are the problems' vectors one after the other (problem p
 * at the sum of the counts before it), tau_dev [n_problems]; each problem is labelled over its own
 * targets, bit-identical to numpy.  bore_is_duplicate_ragged: group g stores n_prev_host[g] >= 0 rows
 * (0 allowed: nothing is a duplicate), x_prev_dev holds the groups' rows one group after the other;
 * x_dev, dup_dev and keep_dev keep the layout of bore_is_duplicate.                                */
int bore_quantile_labels_ragged(const double *y_dev, int n_problems, const int32_t *n_host, double q,
                                float *z_f32_dev, uint8_t *z_u8_dev, double *tau_dev, int device, void *stream);
int bore_is_duplicate_ragged(const double *x_dev, int n_groups, int per_group, const double *x_prev_dev,
                             const int32_t *n_prev_host, int D, double rtol, double atol, uint8_t *dup_dev,
                             uint8_t *keep_dev, int device, void *stream);

/* ---- batch argmax by SVGD (SURVEY.md section 8f, row 3) ---------------------------------
 * Replaces BatchMaximizableMixin.argmax_batch (bore/mixins.py:100-116), i.e.
 * SVGD.optimize_from_init (bore/optimizers/svgd/base.py:78-118) with RadialBasis
 * (svgd/kernels.py:13-28), for n particles per problem, x_dev [n_problems][n][D] fp64 in/out.
 *   length_scale  NaN = None: median heuristic sqrt(.5 * median(r2) / log(n + 1)); floored at 1e-6
 *   lambd         NaN = DistortionConstant(zeta_c); else DistortionExpDecay: rank(f) ** -lambd
 *   step_size, alpha, eps, tau: SVGD.__init__ (svgd/base.py:69-70)
 * bore_svgd_maximize runs n_iter iterations with the handle's model(s) as `func`
 * (transform(model(x)), maximised: `self._func_max`, bore/mixins.py:98) -- two launches per
 * iteration, no host round trip; lo_host / hi_host (both or neither) clip every iterate.
 * bore_svgd_step is ONE iteration for a caller-supplied objective: f_dev [n_problems][n] and
 * g_dev [n_problems][n][D] hold func(x) as fp32 or fp64 (fg_is_f64); `iteration` == 0 starts the
 * AdaGrad accumulator hist_dev [n_problems][n][D]; x32_dev (may be NULL) receives an fp32 copy
 * of the new x.
 * bore_svgd_kernel_value_and_grad is RadialBasis.value_and_grad alone: K [n][n], K_grad [n][D]. */
size_t bore_svgd_workspace_bytes(int n_problems, int n, int D);
int bore_svgd_maximize(bore_mlp *h, int model0, int n_problems, int transform, double *x_dev, int n,
                       const double *lo_host, const double *hi_host, double length_scale, int n_iter,
                       double step_size, double alpha, double eps, double tau, double lambd,
                       double zeta_c, void *work_dev, size_t work_bytes, void *stream);
int bore_svgd_step(double *x_dev, int n_problems, int n, int D, const void *f_dev, const void *g_dev,
                   int fg_is_f64, const double *lo_dev, const double *hi_dev, double length_scale,
                   int iteration, double step_size, double alpha, double eps, double tau, double lambd,
                   double zeta_c, double *hist_dev, float *x32_dev, int device, void *stream);
int bore_svgd_kernel_value_and_grad(const double *x_dev, int n, int D, double length_scale,
                                    double *K_dev, double *Kgrad_dev, int device, void *stream);

/* ---- K7: LSTM multi-fidelity classifier (SURVEY.md section 8f, row 4) --------------------
 * Replaces the Keras networks of StackedRecurrentFactory (bore/models.py:48-104): `num_layers`
 * LSTMCell(units, activation) + Dense(1).  Parameters in Keras get_weights() order
 * [K_0 (in,4U), R_0 (U,4U), b_0 (4U), K_1, R_1, b_1, ..., W_dense (U,1), b_dense (1)], gate order
 * i, f, c, o, recurrent activation sigmoid.  Limits: input_dim <= 32, units <= 32, layers <= 4,
 * steps <= 8, batch <= 64.
 *   bore_lstm_predict_sequences  the many-to-many network (Masking -> RNN... -> TimeDistributed
 *       Dense): X_dev [S][T][D] -> logits out_dev [S][T]; steps whose features ALL equal mask_value
 *       are masked when use_mask != 0 (state and output carried over, keras.backend.rnn).
 *   bore_lstm_predict            the one-to-one network build_one_to_one(num_steps)
 *       (RepeatVector -> same cells -> same Dense on the last step): X_dev [S][D] -> out_dev [S].
 *   bore_lstm_value_and_grad     f = T(+-u(x)), g = df/dx of the one-to-one network -- the convert()
 *       closure (bore/base.py:35-42) that bore_lbfgsb_step is fed with; flags_dev (may be NULL)
 *       selects the rows to evaluate (the stepper's pending flags); X_dev is fp32, or fp64 when
 *       x_is_f64 (the stepper's xreq_dev; rounded to fp32 as Keras casts its input).
 *   bore_lstm_fit                Model.fit on padded sequences (multi_fidelity.py:198-225): X_dev
 *       [N][T][D], Y_dev [N][T], the handle's optimizer (Adam unless bore_lstm_set_optimizer_kind chose
 *       another) + BinaryCrossentropy(from_logits=True) with the mask as sample
 *       weight, divided by batch x steps; perm_dev [epochs][N] int32; loss_dev [epochs].  One launch,
 *       asynchronous on `stream`.
 *   bore_lstm_evaluate           Model.evaluate (multi_fidelity.py:226): out_host[0] = masked loss
 *       (+ l1 / l2 terms), out_host[1] = binary accuracy of the LOGIT at 0.5 over the unmasked steps
 *       (the from_logits quirk; logging only).  Synchronises `stream`.                          */
typedef struct bore_lstm bore_lstm;
int bore_lstm_create(int input_dim, int units, int num_layers, int activation, int device, bore_lstm **out);
int bore_lstm_destroy(bore_lstm *h);
int bore_lstm_num_params(const bore_lstm *h);
int bore_lstm_set_weights(bore_lstm *h, const float *params_host);
int bore_lstm_get_weights(bore_lstm *h, float *params_host);
int bore_lstm_set_adam_state(bore_lstm *h, const float *m_host, const float *v_host, int64_t iterations);
int bore_lstm_get_adam_state(bore_lstm *h, float *m_host, float *v_host, int64_t *iterations);
/* the optimizer and Nadam's momentum cache, as bore_mlp_set_optimizer_kind / bore_mlp_{get,set}_nadam_cache */
int bore_lstm_set_optimizer_kind(bore_lstm *h, int kind, const float *hp);
/* the learning-rate schedule, as bore_mlp_set_lr_schedule */
int bore_lstm_set_lr_schedule(bore_lstm *h, int kind, const float *sp, int n_sp);
int bore_lstm_get_nadam_cache(bore_lstm *h, float *cache_host);
int bore_lstm_set_nadam_cache(bore_lstm *h, float cache);
/* l2 and l1 factors per weight array in Keras order (kernel, recurrent kernel, bias of every cell, then
 * the Dense kernel and bias: 3 * num_layers + 2 floats), as bore_mlp_set_regularizers /
 * bore_mlp_set_l1_regularizers; the l1 factors must be finite and >= 0, and are 0 at create.      */
int bore_lstm_set_regularizers(bore_lstm *h, const float *l2_per_array_host);
int bore_lstm_set_l1_regularizers(bore_lstm *h, const float *l1_per_array_host);
int bore_lstm_predict_sequences(bore_lstm *h, const float *X_dev, int S, int T, float mask_value,
                                int use_mask, float *out_dev, void *stream);
int bore_lstm_predict(bore_lstm *h, const float *X_dev, int S, int num_steps, float *out_dev, void *stream);
int bore_lstm_value_and_grad(bore_lstm *h, int num_steps, int transform, int negate, const void *X_dev,
                             int x_is_f64, int S, const int32_t *flags_dev, float *f_dev, float *g_dev,
                             void *stream);
int bore_lstm_fit(bore_lstm *h, const float *X_dev, const float *Y_dev, int N, int T, float mask_value,
                  int batch_size, int epochs, const int32_t *perm_dev, float *loss_dev, void *stream);
int bore_lstm_evaluate(bore_lstm *h, const float *X_dev, const float *Y_dev, int N, int T, float mask_value,
                       float *out_host, void *stream);

/* ---- measurement helper -----------------------------------------------------------------
 * FP32 FFMA-only microbenchmark (register-resident FMA chains, all SMs): the measured
 * denominator for the FP32 roofline, since MEASURED_PEAKS.json carries only HBM and BF16.
 * Returns TFLOP/s in *tflops_out; synchronous.                                          */
int bore_bench_ffma_peak(int device, int iters, double *tflops_out);

/* ----------------------------------------------------------------------------------------------
 * Host side of the argmax: the candidate points.
 * Replaces `random_state.uniform(low=low, high=high, size=(num_samples, dims))` (bore/mixins.py:49) for a
 * numpy.random.RandomState: the SAME stream (MT19937, 53-bit doubles from two words, low + (high - low) * u)
 * and the same state afterwards, ~5x faster than numpy's broadcasting path -- at configs[2] the draw of
 * 65,536 x 50 doubles per BO iteration took longer than the training kernel.  key[624], *pos: the generator
 * state (RandomState.get_state()[1], [2]), updated on return; low / high: [dim]; out: [n][dim] doubles
 * (any host memory, e.g. the pinned staging buffer of the upload).  Pure host code, no GPU involved.   */
int bore_mt19937_uniform(uint32_t *key, int *pos, const double *low, const double *high, int dim,
                         long long n, double *out);

#ifdef __cplusplus
}
#endif
#endif /* BORE_B200_H */
