// Log-density kernels (SURVEY.md §8 a6, a14, a16, a23) and the LinearCombination predictor (a13).
// Element-wise HBM sweeps with warp-shuffle reductions: one CTA per chain, grid-stride over the elements.
#include "../../include/omc.h"
#include "omc_common.cuh"
#include "omc_internal.h"

namespace {
constexpr int LP_THREADS = 256;
constexpr double LOG_2PI = 1.8378770664093454835606594728112;

__device__ __forceinline__ double vat(const omc_vec_t& v, int chain, long long i, double dflt) {
  return v.ptr ? v.ptr[(long long)chain * v.chain_stride + i] : dflt;
}

__global__ void logp_normal_ss_kernel(omc_logp_normal_ss_t a) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= a.n_chains) return;
  const double s = vat(a.scalar, c, 0, 1.0);
  const double v = 0.5 * (a.dim * log(s) + vat(a.logdet, c, 0, 0.0) - a.dim * LOG_2PI - s * vat(a.ss, c, 0, 0.0));
  a.out[c] = a.accumulate ? a.out[c] + v : v;
}

__global__ void __launch_bounds__(LP_THREADS) logp_gamma_kernel(omc_logp_gamma_t a) {
  __shared__ double scratch[32];
  const int c = blockIdx.x;
  double acc = 0.0;
  for (int i = threadIdx.x; i < a.n_elem; i += LP_THREADS) {
    const double x = vat(a.x, c, i, 0.0);
    const double sh = vat(a.shape, c, a.shape_len > 1 ? i : 0, 1.0);
    const double rt = vat(a.rate, c, a.rate_len > 1 ? i : 0, 1.0);
    const double scale = 1.0 / rt;
    const double y = x / scale;
    double lp = omc_xlogy(sh - 1.0, y) - y - lgamma(sh) - log(scale);
    if (!(sh > 0.0) || rt < 0.0) lp = nan("");               // scipy: invalid shape / rate -> nan
    else if (!(y >= 0.0)) lp = isnan(y) ? y : -INFINITY;
    acc += lp;
  }
  acc = omc_block_sum(acc, scratch);
  if (threadIdx.x == 0) a.out[c] = a.accumulate ? a.out[c] + acc : acc;
}

__global__ void __launch_bounds__(LP_THREADS) logp_poisson_kernel(omc_logp_poisson_t a) {
  __shared__ double scratch[32];
  const int c = blockIdx.x;
  double acc = 0.0;
  for (int i = threadIdx.x; i < a.n_elem; i += LP_THREADS) {
    const double k = vat(a.k, c, i, 0.0);
    const double mu = vat(a.rate, c, a.rate_len > 1 ? i : 0, 1.0);
    double lp = omc_xlogy(k, mu) - lgamma(k + 1.0) - mu;
    if (!(mu >= 0.0)) lp = nan("");                           // scipy: invalid rate -> nan
    else if (!(k >= 0.0) || floor(k) != k) lp = isnan(k) ? k : -INFINITY;   // off the support
    acc += lp;
  }
  acc = omc_block_sum(acc, scratch);
  if (threadIdx.x == 0) a.out[c] = a.accumulate ? a.out[c] + acc : acc;
}

__global__ void logp_const_kernel(double v, int n, double* out, int accumulate) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < n) out[c] = accumulate ? out[c] + v : v;
}

// one warp per output row; rows of X_t are contiguous (p_t doubles)
__global__ void __launch_bounds__(LP_THREADS) linear_predictor_kernel(omc_linear_predictor_t a) {
  const int lane = threadIdx.x & 31;
  const long long warp_global = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  const long long total = (long long)a.n_chains * a.n;
  for (long long row = warp_global; row < total; row += nwarps) {
    const int c = (int)(row / a.n);
    const int r = (int)(row - (long long)c * a.n);
    double acc = 0.0;
    for (int t = 0; t < a.n_terms; ++t) {
      const int p = a.p[t];
      const double* x = a.X[t].ptr + (long long)c * a.X[t].chain_stride + (long long)r * p;
      const double* th = a.theta[t].ptr + (long long)c * a.theta[t].chain_stride;
      if (a.transform_exp[t]) {
        for (int j = lane; j < p; j += 32) acc = fma(x[j], exp(th[j]), acc);
      } else {
        for (int j = lane; j < p; j += 32) acc = fma(x[j], th[j], acc);
      }
    }
    acc = omc_warp_sum(acc);
    if (lane == 0)
      a.out[row] = a.residual_of.ptr ? a.residual_of.ptr[(long long)c * a.residual_of.chain_stride + r] - acc : acc;
  }
}
// Streaming form of the single-term predictor for 2 <= p <= 64, p even (the fitted values X beta of every stored
// iteration, mcmc.py:109-111, and the explicit residual of the re-centring prologue): a warp takes 16 consecutive rows of
// one chain, every lane one 16-byte pair of columns -- the 16 row loads go out together (8 KB in flight per warp), theta
// sits in registers, the 16 row sums are reduced together (first across the two half-warps, then by halving: 31
// double shuffles per 16 rows instead of 5 per row) and leave as one coalesced store.  The generic kernel above re-read
// theta per row, reduced every row on its own and stored 8 bytes per warp and row: 2.1 TB/s on the C2 shape.
constexpr int LPR_ROWS = 16;
__global__ void __launch_bounds__(LP_THREADS) linear_predictor_rows_kernel(omc_linear_predictor_t a) {
  const int lane = threadIdx.x & 31;
  const int p = a.p[0];
  const long long blocks_per_chain = (a.n + LPR_ROWS - 1) / LPR_ROWS;
  const long long total = (long long)a.n_chains * blocks_per_chain;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  const bool live = 2 * lane < p;
  for (long long blk = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; blk < total; blk += nwarps) {
    const int c = (int)(blk / blocks_per_chain);
    const long long r0 = (blk - (long long)c * blocks_per_chain) * LPR_ROWS;
    const double* th = a.theta[0].ptr + (long long)c * a.theta[0].chain_stride;
    double t0 = live ? th[2 * lane] : 0.0, t1 = live ? th[2 * lane + 1] : 0.0;
    if (a.transform_exp[0]) { t0 = live ? exp(t0) : 0.0; t1 = live ? exp(t1) : 0.0; }
    const double* x = a.X[0].ptr + (long long)c * a.X[0].chain_stride + r0 * p + 2 * lane;
    double2 xv[LPR_ROWS];
#pragma unroll
    for (int i = 0; i < LPR_ROWS; ++i)
      xv[i] = (live && r0 + i < a.n) ? __ldg(reinterpret_cast<const double2*>(x + (long long)i * p)) : make_double2(0.0, 0.0);
    double v[LPR_ROWS];
#pragma unroll
    for (int i = 0; i < LPR_ROWS; ++i) v[i] = fma(xv[i].x, t0, xv[i].y * t1);
    // lanes l and l ^ 16 first (all 16 sums), then keep half of the sums per step: lane l ends with row (l & 15)
#pragma unroll
    for (int i = 0; i < LPR_ROWS; ++i) v[i] += omc_shfl_xor(v[i], 16);
#pragma unroll
    for (int h = 8; h >= 1; h >>= 1) {
      const bool upper = (lane & h) != 0;
#pragma unroll
      for (int i = 0; i < h; ++i) {
        const double keep = upper ? v[i + h] : v[i], send = upper ? v[i] : v[i + h];
        v[i] = keep + omc_shfl_xor(send, h);
      }
    }
    const long long r = r0 + (lane & 15);
    if (lane < 16 && r < a.n) {
      const long long o = (long long)c * a.n + r;
      a.out[o] = a.residual_of.ptr ? a.residual_of.ptr[(long long)c * a.residual_of.chain_stride + r] - v[0] : v[0];
    }
  }
}
__global__ void __launch_bounds__(LP_THREADS) sum_log_kernel(const double* x, long long n, double* out) {
  __shared__ double scratch[32];
  const double* xm = x + (long long)blockIdx.x * n;
  double acc = 0.0;
  for (long long i = threadIdx.x; i < n; i += LP_THREADS) acc += log(xm[i]);
  acc = omc_block_sum(acc, scratch);
  if (threadIdx.x == 0) out[blockIdx.x] = acc;
}

// out = log(x), element-wise (the log-response of a LogNormal whose response is data: location_scale.py:296-303)
__global__ void __launch_bounds__(LP_THREADS) log_elements_kernel(const double* x, long long n, double* out) {
  for (long long i = (long long)blockIdx.x * LP_THREADS + threadIdx.x; i < n; i += (long long)gridDim.x * LP_THREADS)
    out[i] = log(x[i]);
}

// unblocked Cholesky of one small matrix per CTA (setup-time only)
__global__ void __launch_bounds__(64) logdet_dense_kernel(const double* P, int n, double* out) {
  extern __shared__ double A[];
  const double* Pm = P + (long long)blockIdx.x * n * n;
  const int tid = threadIdx.x;
  for (int e = tid; e < n * n; e += 64) A[e] = Pm[e];
  __syncthreads();
  double ld = 0.0;
  for (int j = 0; j < n; ++j) {
    const double d = A[j * n + j];
    if (!(d > 0.0)) { ld = nan(""); break; }
    const double s = sqrt(d);
    ld += 2.0 * log(s);
    __syncthreads();
    for (int i = j + 1 + tid; i < n; i += 64) A[i * n + j] /= s;
    __syncthreads();
    for (int i = j + 1 + tid; i < n; i += 64)
      for (int c = j + 1; c <= i; ++c) A[i * n + c] -= A[i * n + j] * A[c * n + j];
    __syncthreads();
  }
  if (tid == 0) out[blockIdx.x] = ld;
}
// out[c][i] = sum_t scale_t[c] * x_t[c][i]  (t < n_terms <= 4; scale NULL => 1)
__global__ void combine_kernel(int n_chains, long long len, int n_terms, omc_vec_t x0, omc_vec_t x1, omc_vec_t x2,
                               omc_vec_t x3, omc_vec_t s0, omc_vec_t s1, omc_vec_t s2, omc_vec_t s3, double* out) {
  const long long total = (long long)n_chains * len;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(e / len);
    const long long i = e - (long long)c * len;
    double v = vat(s0, c, 0, 1.0) * vat(x0, c, i, 0.0);
    if (n_terms > 1) v = fma(vat(s1, c, 0, 1.0), vat(x1, c, i, 0.0), v);
    if (n_terms > 2) v = fma(vat(s2, c, 0, 1.0), vat(x2, c, i, 0.0), v);
    if (n_terms > 3) v = fma(vat(s3, c, 0, 1.0), vat(x3, c, i, 0.0), v);
    out[e] = v;
  }
}
__global__ void logp_domain_kernel(int n_chains, int n_elem, omc_vec_t x, omc_vec_t lower, int lo_len, omc_vec_t upper,
                                   int hi_len, double* out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_chains) return;
  bool outside = false;
  for (int i = 0; i < n_elem; ++i) {
    const double v = x.ptr[(long long)c * x.chain_stride + i];
    if (lower.ptr && v < lower.ptr[(long long)c * lower.chain_stride + (lo_len > 1 ? i : 0)]) outside = true;
    if (upper.ptr && v > upper.ptr[(long long)c * upper.chain_stride + (hi_len > 1 ? i : 0)]) outside = true;
  }
  if (outside) out[c] = -INFINITY;
}
}  // namespace

extern "C" {
int omc_sum_log(const double* x, int n_mats, long long n, double* out, void* stream) {
  OMC_REQUIRE(x && out && n_mats >= 1 && n >= 0, "omc_sum_log: bad argument");
  sum_log_kernel<<<n_mats, LP_THREADS, 0, (cudaStream_t)stream>>>(x, n, out);
  OMC_LAUNCH_CHECK();
  return 0;
}
int omc_log_elements(const double* x, long long n, double* out, void* stream) {
  OMC_REQUIRE(x && out && n >= 1, "omc_log_elements: bad argument");
  const long long blocks = (n + LP_THREADS - 1) / LP_THREADS;
  log_elements_kernel<<<(unsigned)(blocks < 4096 ? blocks : 4096), LP_THREADS, 0, (cudaStream_t)stream>>>(x, n, out);
  OMC_LAUNCH_CHECK();
  return 0;
}
int omc_logdet_dense(const double* P, int n_mats, int n, double* out, void* stream) {
  OMC_REQUIRE(P && out && n_mats >= 1 && n >= 1 && n <= 64, "omc_logdet_dense: bad argument (n=%d)", n);
  logdet_dense_kernel<<<n_mats, 64, (size_t)n * n * sizeof(double), (cudaStream_t)stream>>>(P, n, out);
  OMC_LAUNCH_CHECK();
  return 0;
}
int omc_logp_normal_ss(const omc_logp_normal_ss_t* a, void* stream) {
  OMC_REQUIRE(a && a->out && a->ss.ptr, "omc_logp_normal_ss: null argument");
  logp_normal_ss_kernel<<<(a->n_chains + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*a);
  OMC_LAUNCH_CHECK();
  return 0;
}
int omc_logp_gamma(const omc_logp_gamma_t* a, void* stream) {
  OMC_REQUIRE(a && a->out && (a->x.ptr || a->n_elem == 0), "omc_logp_gamma: null argument");
  OMC_REQUIRE(a->n_chains >= 1 && a->n_elem >= 0, "omc_logp_gamma: bad shape");
  logp_gamma_kernel<<<a->n_chains, LP_THREADS, 0, (cudaStream_t)stream>>>(*a);
  OMC_LAUNCH_CHECK();
  return 0;
}
int omc_logp_poisson(const omc_logp_poisson_t* a, void* stream) {
  OMC_REQUIRE(a && a->out && (a->k.ptr || a->n_elem == 0), "omc_logp_poisson: null argument");
  OMC_REQUIRE(a->n_chains >= 1 && a->n_elem >= 0, "omc_logp_poisson: bad shape");
  logp_poisson_kernel<<<a->n_chains, LP_THREADS, 0, (cudaStream_t)stream>>>(*a);
  OMC_LAUNCH_CHECK();
  return 0;
}
int omc_logp_const(double value, int n_chains, double* out, int accumulate, void* stream) {
  OMC_REQUIRE(out && n_chains >= 1, "omc_logp_const: bad argument");
  logp_const_kernel<<<(n_chains + 127) / 128, 128, 0, (cudaStream_t)stream>>>(value, n_chains, out, accumulate);
  OMC_LAUNCH_CHECK();
  return 0;
}
int omc_logp_domain(int n_chains, int n_elem, omc_vec_t x, omc_vec_t lower, int lo_len, omc_vec_t upper, int hi_len,
                    double* out, void* stream) {
  OMC_REQUIRE(out && x.ptr && n_chains >= 1 && n_elem >= 1, "omc_logp_domain: bad argument");
  logp_domain_kernel<<<(n_chains + 127) / 128, 128, 0, (cudaStream_t)stream>>>(n_chains, n_elem, x, lower, lo_len, upper,
                                                                              hi_len, out);
  OMC_LAUNCH_CHECK();
  return 0;
}
int omc_combine(int n_chains, long long len, int n_terms, const omc_vec_t* x, const omc_vec_t* scale, double* out,
                void* stream) {
  OMC_REQUIRE(out && x && n_chains >= 1 && len >= 0 && n_terms >= 1 && n_terms <= 4, "omc_combine: bad argument");
  if (len == 0) return 0;
  const omc_vec_t none = {nullptr, 0};
  omc_vec_t xs[4], ss[4];
  for (int t = 0; t < 4; ++t) {
    xs[t] = t < n_terms ? x[t] : none;
    ss[t] = (t < n_terms && scale) ? scale[t] : none;
    OMC_REQUIRE(t >= n_terms || xs[t].ptr, "omc_combine: term %d is NULL", t);
  }
  const long long total = (long long)n_chains * len;
  long long blocks = (total + 255) / 256;
  const long long cap = (long long)omc_sm_count() * 16;
  if (blocks > cap) blocks = cap;
  combine_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(n_chains, len, n_terms, xs[0], xs[1], xs[2], xs[3], ss[0],
                                                                     ss[1], ss[2], ss[3], out);
  OMC_LAUNCH_CHECK();
  return 0;
}
int omc_linear_predictor(const omc_linear_predictor_t* a, void* stream) {
  OMC_REQUIRE(a && a->out && a->n_terms >= 1 && a->n_terms <= 4, "omc_linear_predictor: bad argument");
  const long long total = (long long)a->n_chains * a->n;
  const long long cap = (long long)omc_sm_count() * 16;
  const int p0 = a->p[0];
  if (a->n_terms == 1 && p0 >= 2 && p0 <= 64 && p0 % 2 == 0 && a->X[0].ptr && a->theta[0].ptr &&
      (reinterpret_cast<uintptr_t>(a->X[0].ptr) & 15) == 0 && a->X[0].chain_stride % 2 == 0) {
    long long blocks = ((total + LPR_ROWS - 1) / LPR_ROWS * 32 + LP_THREADS - 1) / LP_THREADS;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    linear_predictor_rows_kernel<<<(unsigned)blocks, LP_THREADS, 0, (cudaStream_t)stream>>>(*a);
    OMC_LAUNCH_CHECK();
    return 0;
  }
  long long blocks = (total * 32 + LP_THREADS - 1) / LP_THREADS;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  linear_predictor_kernel<<<(unsigned)blocks, LP_THREADS, 0, (cudaStream_t)stream>>>(*a);
  OMC_LAUNCH_CHECK();
  return 0;
}
}
