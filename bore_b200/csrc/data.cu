// Data step either side of the hot path (SURVEY.md section 8f row 2), sm_100a.
//
//  * bore_quantile_labels   replaces Record.load_classification_data (bore/data.py:31-35):
//    tau = np.quantile(y, q=gamma) (method "linear"), z = np.less(y, tau) -- for M problems at
//    once, one CTA per problem, so that a batched BO iteration (BASELINE.json configs[3]) feeds
//    raw targets to the GPU and the labels never exist on the host.
//  * bore_is_duplicate      replaces Record.is_duplicate (bore/data.py:42-48):
//    any(np.allclose(x_prev, x, rtol, atol) for x_prev in features) for every candidate x of a
//    group against that group's stored observations; its output is the `keep` mask of
//    bore_select_best / bore_select_best_groups, i.e. the plugin's filter_fn=_is_unique
//    (bore/plugins/hpbandster/base.py:227-231, 264) evaluated for all results in one launch.
//
// Both are exact fp64 / integer work (no FMA contraction: numpy rounds every product and sum),
// bit-identical to numpy on finite input.
#include <algorithm>

#include "common.cuh"

namespace {

// monotone map double -> uint64 (ascending); -0 and +0 map to the same key, NaN sorts last
__device__ __forceinline__ unsigned long long orderable64(double v) {
  if (v != v) return ~0ULL - 1ULL;  // below the padding key, above every number
  if (v == 0.0) v = 0.0;
  const unsigned long long u = (unsigned long long)__double_as_longlong(v);
  return (u >> 63) ? ~u : (u | 0x8000000000000000ULL);
}
__device__ __forceinline__ double from_orderable64(unsigned long long k) {
  const unsigned long long u = (k >> 63) ? (k & 0x7fffffffffffffffULL) : ~k;
  return __longlong_as_double((long long)u);
}

__host__ __device__ int pow2_at_least(int v) { int p = 1; while (p < v) p <<= 1; return p; }

// one CTA per problem: keys of the N targets sorted in shared memory (bitonic, padded to a power
// of two), the two order statistics around the virtual index (N-1)*q read off, numpy's _lerp
// applied, labels written as fp32 0/1 (what fit consumes) and/or bytes.  `off` (ragged problems;
// NULL: every problem holds N targets): problem b is y[off[b], off[b+1]); its CTA sorts its own
// power of two inside shared memory sized for the largest.
__global__ void __launch_bounds__(1024)
quantile_labels_kernel(const double *__restrict__ y, const long long *__restrict__ off, int N, int n_pow2,
                       double q, float *__restrict__ z_f32, uint8_t *__restrict__ z_u8,
                       double *__restrict__ tau_out) {
  extern __shared__ unsigned long long sk[];
  __shared__ double s_tau;
  __shared__ int s_nan;
  long long o0 = (long long)blockIdx.x * N;
  if (off) {
    o0 = off[blockIdx.x];
    N = (int)(off[blockIdx.x + 1] - o0);
    n_pow2 = max(2, pow2_at_least(N));
  }
  const double *yp = y + o0;
  if (threadIdx.x == 0) s_nan = 0;
  __syncthreads();
  bool has_nan = false;
  for (int i = threadIdx.x; i < n_pow2; i += blockDim.x) {
    unsigned long long key = ~0ULL;
    if (i < N) {
      const double v = yp[i];
      has_nan |= (v != v);
      key = orderable64(v);
    }
    sk[i] = key;
  }
  if (has_nan) s_nan = 1;
  __syncthreads();
  for (int kk = 2; kk <= n_pow2; kk <<= 1)
    for (int j = kk >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < n_pow2; i += blockDim.x) {
        const int ixj = i ^ j;
        if (ixj > i) {
          const unsigned long long a = sk[i], b = sk[ixj];
          const bool up = (i & kk) == 0;
          if ((a > b) == up) { sk[i] = b; sk[ixj] = a; }
        }
      }
      __syncthreads();
    }
  if (threadIdx.x == 0) {
    // numpy/lib/_function_base_impl.py::_quantile, method "linear": virtual index (N-1)*q,
    // neighbours floor / floor+1 (clamped at the ends), gamma = the fractional part, then
    // _lerp(a, b, t) = a + (b-a)*t, replaced by b - (b-a)*(1-t) where t >= 0.5
    double tau;
    if (s_nan) {
      tau = __longlong_as_double(0x7ff8000000000000LL);  // a slice holding NaN yields NaN
    } else {
      const double vi = __dmul_rn((double)(N - 1), q);
      int prev, next;
      double t;
      if (vi >= (double)(N - 1)) { prev = next = N - 1; t = 0.0; }
      else if (vi < 0.0) { prev = next = 0; t = 0.0; }
      else { const double fl = floor(vi); prev = (int)fl; next = prev + 1; t = __dsub_rn(vi, fl); }
      const double a = from_orderable64(sk[prev]), b = from_orderable64(sk[next]);
      const double diff = __dsub_rn(b, a);
      tau = (t >= 0.5) ? __dsub_rn(b, __dmul_rn(diff, __dsub_rn(1.0, t)))
                       : __dadd_rn(a, __dmul_rn(diff, t));
    }
    s_tau = tau;
    if (tau_out) tau_out[blockIdx.x] = tau;
  }
  __syncthreads();
  const double tau = s_tau;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    const bool z = yp[i] < tau;  // STRICT (np.less); false against a NaN threshold
    if (z_f32) z_f32[o0 + i] = z ? 1.f : 0.f;
    if (z_u8) z_u8[o0 + i] = z ? 1 : 0;
  }
}

// one warp per candidate: lanes walk the stored rows of the candidate's group; a row matches
// when every coordinate satisfies numpy.isclose(a = x_prev, b = x):
//   |a - b| <= atol + rtol * |b|  and b finite,  or  a == b
// `off` (ragged groups; NULL: every group stores n_prev rows): group g's rows are [off[g], off[g+1])
__global__ void __launch_bounds__(256)
duplicate_kernel(const double *__restrict__ x, int n_groups, int per_group,
                 const double *__restrict__ x_prev, const long long *__restrict__ off, int n_prev, int D,
                 double rtol, double atol, uint8_t *__restrict__ dup_out, uint8_t *__restrict__ keep_out) {
  const int cand = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (cand >= n_groups * per_group) return;
  const int g = cand / per_group;
  const double *xc = x + (size_t)cand * D;
  long long r0 = (long long)g * n_prev;
  if (off) {
    r0 = off[g];
    n_prev = (int)(off[g + 1] - r0);
  }
  const double *xp = x_prev + r0 * D;
  bool found = false;
  for (int r0 = 0; r0 < n_prev && !found; r0 += 32) {
    const int r = r0 + lane;
    bool all = r < n_prev;
    for (int d = 0; d < D && all; ++d) {
      const double a = xp[(size_t)r * D + d], b = xc[d];
      const bool close = fabs(__dsub_rn(a, b)) <= __dadd_rn(atol, __dmul_rn(rtol, fabs(b)));
      all = (close && isfinite(b)) || a == b;
    }
    found = __any_sync(0xffffffffu, all);
  }
  if (lane == 0) {
    if (dup_out) dup_out[cand] = found ? 1 : 0;
    if (keep_out) keep_out[cand] = found ? 0 : 1;
  }
}

// maybe_distort (bore/base.py:45-64): x = truncnorm(a, b, loc, scale).rvs(random_state) with
// a = (lower - loc) / scale, b = (upper - loc) / scale.  scipy draws ONE uniform variate per
// coordinate from the caller's MT19937 stream and maps it through the distribution's ppf; the
// variates are drawn on the host (stream parity) and uploaded, the ppf runs here:
//   a <  0:  x =  ndtri(Phi(a)  + q       * mass)
//   a >= 0:  x = -ndtri(Phi(-b) + (1 - q) * mass)        (right tail through the survival side)
// with mass = Phi(b) - Phi(a) taken on the side where it does not cancel -- scipy's case split
// (scipy/stats/_continuous_distns.py, truncnorm_gen._ppf / _log_gauss_mass) without the detour
// through logarithms, which only matters for intervals deep in one tail (loc lies inside the box
// here).  One thread per coordinate.
__global__ void __launch_bounds__(256)
truncnorm_distort_kernel(const double *__restrict__ loc, long n_total, int D, double scale,
                         const double *__restrict__ lo, const double *__restrict__ hi,
                         const double *__restrict__ u, double *__restrict__ out) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_total) return;
  const int d = (int)(i % D);
  const double l = loc[i], q = u[i];
  const double a = (lo[d] - l) / scale, b = (hi[d] - l) / scale;
  double mass;
  if (b <= 0.0) mass = normcdf(b) - normcdf(a);
  else if (a > 0.0) mass = normcdf(-a) - normcdf(-b);
  else mass = 1.0 - normcdf(a) - normcdf(-b);
  double x;
  if (a < 0.0) x = normcdfinv(normcdf(a) + q * mass);
  else x = -normcdfinv(normcdf(-b) + (1.0 - q) * mass);
  // the standardised variate lies in [a, b] up to rounding: clamp like the support does
  x = fmin(fmax(x, a), b);
  out[i] = l + scale * x;
}

}  // namespace

// bore_quantile_labels and its ragged form: N the (largest) number of targets, off_host (ragged; may be NULL)
// the n_problems + 1 offsets of the problems in y
static int quantile_run(const double *y_dev, int n_problems, const long long *off_host, int N, double q,
                        float *z_f32_dev, uint8_t *z_u8_dev, double *tau_dev, int device, void *stream_) {
  BORE_CHECK(q >= 0.0 && q <= 1.0, "Quantiles must be in the range [0, 1]");  // numpy's message
  BORE_CHECK(y_dev && (z_f32_dev || z_u8_dev || tau_dev), "bore_quantile_labels: NULL buffer");
  const int n = std::max(2, pow2_at_least(N));
  const size_t smem = (size_t)n * sizeof(unsigned long long);
  BORE_CHECK(smem <= 224 * 1024, "bore_quantile_labels: N=%d exceeds the shared-memory sort (max 16384)", N);
  BORE_CUDA(cudaSetDevice(device));
  static bool attr_done[64] = {};
  if (device >= 64 || !attr_done[device]) {
    BORE_CUDA(cudaFuncSetAttribute(quantile_labels_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   224 * 1024));
    if (device < 64) attr_done[device] = true;
  }
  const cudaStream_t stream = (cudaStream_t)stream_;
  StreamTable table;  // freed on the stream after the launch
  if (off_host) BORE_CUDA(table.upload(off_host, (size_t)(n_problems + 1) * sizeof(long long), stream));
  const int threads = std::min(1024, std::max(32, n / 2));
  quantile_labels_kernel<<<n_problems, threads, smem, stream>>>(y_dev, static_cast<const long long *>(table.dev),
                                                                N, n, q, z_f32_dev, z_u8_dev, tau_dev);
  BORE_CUDA(cudaGetLastError());
  return 0;
}

// bore_is_duplicate and its ragged form: off_host (ragged; may be NULL) the n_groups + 1 offsets of the groups'
// stored rows in x_prev, any_prev whether there is a stored row at all
static int duplicate_run(const double *x_dev, int n_groups, int per_group, const double *x_prev_dev,
                         const long long *off_host, int n_prev, bool any_prev, int D, double rtol, double atol,
                         uint8_t *dup_dev, uint8_t *keep_dev, int device, void *stream_) {
  BORE_CHECK(x_dev && (!any_prev || x_prev_dev) && (dup_dev || keep_dev), "bore_is_duplicate: NULL buffer");
  BORE_CUDA(cudaSetDevice(device));
  const cudaStream_t stream = (cudaStream_t)stream_;
  StreamTable table;  // freed on the stream after the launch
  if (off_host) BORE_CUDA(table.upload(off_host, (size_t)(n_groups + 1) * sizeof(long long), stream));
  const long warps = (long)n_groups * per_group;
  const int blocks = (int)((warps * 32 + 255) / 256);
  duplicate_kernel<<<blocks, 256, 0, stream>>>(x_dev, n_groups, per_group, x_prev_dev,
                                               static_cast<const long long *>(table.dev), n_prev, D, rtol, atol,
                                               dup_dev, keep_dev);
  BORE_CUDA(cudaGetLastError());
  return 0;
}

extern "C" {

int bore_quantile_labels(const double *y_dev, int n_problems, int N, double q, float *z_f32_dev,
                         uint8_t *z_u8_dev, double *tau_dev, int device, void *stream_) {
  BORE_CHECK(bore_device_count() > 0, "no CUDA device visible -- bore_b200 has no CPU fallback");
  BORE_CHECK(n_problems >= 1 && N >= 1, "bore_quantile_labels: n_problems=%d, N=%d", n_problems, N);
  return quantile_run(y_dev, n_problems, nullptr, N, q, z_f32_dev, z_u8_dev, tau_dev, device, stream_);
}

int bore_quantile_labels_ragged(const double *y_dev, int n_problems, const int32_t *n_host, double q,
                                float *z_f32_dev, uint8_t *z_u8_dev, double *tau_dev, int device, void *stream_) {
  BORE_CHECK(bore_device_count() > 0, "no CUDA device visible -- bore_b200 has no CPU fallback");
  BORE_CHECK(n_problems >= 1 && n_host, "bore_quantile_labels_ragged: n_problems=%d, n_host=%p", n_problems,
             (const void *)n_host);
  std::vector<long long> off(n_problems + 1, 0);
  int maxN = 1;
  for (int p = 0; p < n_problems; ++p) {
    // N_p <= 16384 is checked below (through the largest), so the sum cannot overflow
    BORE_CHECK(n_host[p] >= 1, "bore_quantile_labels_ragged: problem %d has N=%d", p, n_host[p]);
    off[p + 1] = off[p] + n_host[p];
    maxN = std::max(maxN, (int)n_host[p]);
  }
  return quantile_run(y_dev, n_problems, off.data(), maxN, q, z_f32_dev, z_u8_dev, tau_dev, device, stream_);
}

int bore_is_duplicate(const double *x_dev, int n_groups, int per_group, const double *x_prev_dev,
                      int n_prev, int D, double rtol, double atol, uint8_t *dup_dev,
                      uint8_t *keep_dev, int device, void *stream_) {
  BORE_CHECK(bore_device_count() > 0, "no CUDA device visible -- bore_b200 has no CPU fallback");
  BORE_CHECK(n_groups >= 1 && per_group >= 1 && n_prev >= 0 && D >= 1,
             "bore_is_duplicate: n_groups=%d, per_group=%d, n_prev=%d, D=%d", n_groups, per_group,
             n_prev, D);
  return duplicate_run(x_dev, n_groups, per_group, x_prev_dev, nullptr, n_prev, n_prev > 0, D, rtol, atol,
                       dup_dev, keep_dev, device, stream_);
}

int bore_is_duplicate_ragged(const double *x_dev, int n_groups, int per_group, const double *x_prev_dev,
                             const int32_t *n_prev_host, int D, double rtol, double atol, uint8_t *dup_dev,
                             uint8_t *keep_dev, int device, void *stream_) {
  BORE_CHECK(bore_device_count() > 0, "no CUDA device visible -- bore_b200 has no CPU fallback");
  BORE_CHECK(n_groups >= 1 && per_group >= 1 && D >= 1 && n_prev_host,
             "bore_is_duplicate_ragged: n_groups=%d, per_group=%d, D=%d, n_prev_host=%p", n_groups, per_group, D,
             (const void *)n_prev_host);
  BORE_CHECK((long long)n_groups * per_group <= 0x7fffffffLL / 32,
             "bore_is_duplicate_ragged: %d x %d candidates", n_groups, per_group);
  std::vector<long long> off(n_groups + 1, 0);
  for (int g = 0; g < n_groups; ++g) {
    BORE_CHECK(n_prev_host[g] >= 0, "bore_is_duplicate_ragged: group %d has n_prev=%d", g, n_prev_host[g]);
    off[g + 1] = off[g] + n_prev_host[g];  // < 2^31 * 2^31: no overflow
  }
  BORE_CHECK(off[n_groups] <= 0x7fffffffffffffffLL / D, "bore_is_duplicate_ragged: the stored rows overflow 64 bits");
  return duplicate_run(x_dev, n_groups, per_group, x_prev_dev, off.data(), 0, off[n_groups] > 0, D, rtol, atol,
                       dup_dev, keep_dev, device, stream_);
}

int bore_truncnorm_distort(const double *loc_dev, int n_points, int D, double scale,
                           const double *lo_dev, const double *hi_dev, const double *u_dev,
                           double *out_dev, int device, void *stream_) {
  BORE_CHECK(bore_device_count() > 0, "no CUDA device visible -- bore_b200 has no CPU fallback");
  BORE_CHECK(n_points >= 1 && D >= 1, "bore_truncnorm_distort: n_points=%d, D=%d", n_points, D);
  BORE_CHECK(scale > 0.0, "bore_truncnorm_distort: scale must be positive");
  BORE_CHECK(loc_dev && lo_dev && hi_dev && u_dev && out_dev, "bore_truncnorm_distort: NULL buffer");
  BORE_CUDA(cudaSetDevice(device));
  const long n_total = (long)n_points * D;
  truncnorm_distort_kernel<<<(int)((n_total + 255) / 256), 256, 0, (cudaStream_t)stream_>>>(
      loc_dev, n_total, D, scale, lo_dev, hi_dev, u_dev, out_dev);
  BORE_CUDA(cudaGetLastError());
  return 0;
}

}  // extern "C"
