// Metropolis-Hastings kernels (SURVEY.md §8 a5, a6, a14-a21): model log-density / gradient / Hessian over a term list,
// RandomWalk / RandomWalkLoop (Gaussian and truncated-Gaussian proposals) and ManifoldMALA, batched over chains.
//
// Mapping: one WARP per chain for log_p / gradients / random-walk steps (lanes stride over the n_elem parameters, warp
// shuffles reduce the sums); one CTA per chain for ManifoldMALA (dense Hessian + Cholesky in shared memory).  Chain
// state stays in HBM between sweeps; within a kernel it lives in shared memory.  These kernels are latency / FP64-ALU
// bound (lgamma, log, erfc): bytes per chain-iteration are ~1 KB (DESIGN.md).
#include "../../include/omc.h"
#include "omc_common.cuh"
#include "omc_internal.h"
#include "omc_smallmat.cuh"
#include "omc_special.cuh"

namespace {

constexpr double LOG_2PI = 1.8378770664093454835606594728112;
constexpr int MH_WARPS = 4;  // warps (= chains) per CTA in the warp-per-chain kernels

__device__ __forceinline__ double vat(const omc_vec_t& v, int chain, long long i, double dflt) {
  return v.ptr ? v.ptr[(long long)chain * v.chain_stride + i] : dflt;
}
__device__ __forceinline__ OmcRng to_rng(const omc_rng_t& r) {
  OmcRng o;
  o.seed = r.seed; o.sweep = r.sweep; o.chain_offset = r.chain_offset; o.site = r.site;
  return o;
}
__device__ __forceinline__ double mat_at(int kind, const omc_vec_t& P, int chain, int n, int i, int j) {
  if (kind == OMC_MAT_DENSE) return P.ptr[(long long)chain * P.chain_stride + (long long)i * n + j];
  if (i != j) return 0.0;
  if (kind == OMC_MAT_DIAG) return P.ptr[(long long)chain * P.chain_stride + i];
  return P.ptr ? P.ptr[(long long)chain * P.chain_stride] : 1.0;
}

// ---------------------------------------------------------------------------------------------- term log-densities
// Warp-cooperative: every lane of the warp calls with the same arguments; result valid in all lanes.
__device__ double term_logp_warp(const omc_term_t& t, int n, int chain, const double* th) {
  const int lane = threadIdx.x & 31;
  double acc = 0.0;
  switch (t.kind) {
    case OMC_TERM_POISSON_RATE:
      for (int i = lane; i < n; i += 32) {
        const double k = vat(t.data, chain, i, 0.0), mu = th[i];
        double lp = omc_xlogy(k, mu) - lgamma(k + 1.0) - mu;
        if (!(mu >= 0.0)) lp = nan("");                       // scipy: invalid rate -> nan
        else if (!(k >= 0.0) || floor(k) != k) lp = -INFINITY;  // off the support
        acc += lp;
      }
      break;
    case OMC_TERM_GAMMA_RESPONSE:
      for (int i = lane; i < n; i += 32) {
        const double x = th[i];
        const double sh = vat(t.p1, chain, t.p1_len > 1 ? i : 0, 1.0), rt = vat(t.p2, chain, t.p2_len > 1 ? i : 0, 1.0);
        const double scale = 1.0 / rt, y = x / scale;
        double lp = omc_xlogy(sh - 1.0, y) - y - lgamma(sh) - log(scale);
        if (!(y >= 0.0)) lp = isnan(y) ? y : -INFINITY;
        acc += lp;
      }
      break;
    case OMC_TERM_NORMAL_RESPONSE: {
      const double s = vat(t.scalar, chain, 0, 1.0);
      bool outside = false;
      for (int i = lane; i < n; i += 32) {
        const double ri = th[i] - vat(t.p1, chain, t.p1_len > 1 ? i : 0, 0.0);
        if (th[i] < t.dom_lo || th[i] > t.dom_hi) outside = true;
        double q;
        if (t.mat_kind == OMC_MAT_DENSE) {
          q = 0.0;
          for (int j = 0; j < n; ++j)
            q += mat_at(OMC_MAT_DENSE, t.P, chain, n, i, j) * (th[j] - vat(t.p1, chain, t.p1_len > 1 ? j : 0, 0.0));
        } else {
          q = mat_at(t.mat_kind, t.P, chain, n, i, i) * ri;
        }
        acc += ri * q;
      }
      acc = omc_warp_sum(acc);
      outside = __any_sync(0xffffffffu, outside);
      if (outside) return -INFINITY;
      return 0.5 * (n * log(s) + vat(t.logdet, chain, 0, 0.0) - n * LOG_2PI - s * acc);
    }
    case OMC_TERM_UNIFORM_RESPONSE:
      for (int i = lane; i < n; i += 32)
        acc -= log(vat(t.p2, chain, t.p2_len > 1 ? i : 0, 1.0) - vat(t.p1, chain, t.p1_len > 1 ? i : 0, 0.0));
      break;
    case OMC_TERM_LOGNORMAL_RESPONSE: {
      // MVN log-pdf at log(theta) minus sum log(theta) (location_scale.py:296-303); theta <= 0 gives NaN / -inf as numpy
      const double s = vat(t.scalar, chain, 0, 1.0);
      double sumlog = 0.0;
      for (int i = lane; i < n; i += 32) {
        const double li = log(th[i]);
        const double ri = li - vat(t.p1, chain, t.p1_len > 1 ? i : 0, 0.0);
        double q;
        if (t.mat_kind == OMC_MAT_DENSE) {
          q = 0.0;
          for (int j = 0; j < n; ++j)
            q += mat_at(OMC_MAT_DENSE, t.P, chain, n, i, j) * (log(th[j]) - vat(t.p1, chain, t.p1_len > 1 ? j : 0, 0.0));
        } else {
          q = mat_at(t.mat_kind, t.P, chain, n, i, i) * ri;
        }
        acc += ri * q;
        sumlog += li;
      }
      acc = omc_warp_sum(acc);
      sumlog = omc_warp_sum(sumlog);
      return 0.5 * (n * log(s) + vat(t.logdet, chain, 0, 0.0) - n * LOG_2PI - s * acc) - sumlog;
    }
    case OMC_TERM_NORMAL_LINEAR: {
      const double s = vat(t.scalar, chain, 0, 1.0);
      const double* rec = t.stats.ptr + (long long)chain * t.stats.chain_stride;
      const double* G = rec;
      const double* gv = rec + n * n;
      for (int j = lane; j < n; j += 32) {
        double gf = 0.0;
        for (int k = 0; k < n; ++k) gf = fma(G[j * n + k], t.transform_exp ? exp(th[k]) : th[k], gf);
        const double fj = t.transform_exp ? exp(th[j]) : th[j];
        acc = fma(fj, gf - 2.0 * gv[j], acc);
      }
      const double S = rec[n * n + n] + omc_warp_sum(acc);
      return 0.5 * (t.n_data * log(s) + vat(t.logdet, chain, 0, 0.0) - t.n_data * LOG_2PI - s * S);
    }
    default:
      break;
  }
  return omc_warp_sum(acc);
}

__device__ double model_logp_warp(const omc_mh_model_t& m, int chain, const double* th) {
  double s = 0.0;
  for (int k = 0; k < m.n_terms; ++k) s += term_logp_warp(m.terms[k], m.n_elem, chain, th);
  return s;
}

// ---------------------------------------------------------------------------------------------- derivatives
// Analytic gradient (positive log-pdf) and Hessian (negative log-pdf) of one term, accumulated into g[n], H[n x ldh].
// Thread-parallel over `nthr` cooperating threads with index `tid`.
__device__ void term_grad_hess_analytic(const omc_term_t& t, int n, int chain, const double* th, double* g, double* H,
                                        int ldh, int tid, int nthr) {
  switch (t.kind) {
    case OMC_TERM_POISSON_RATE:
      for (int i = tid; i < n; i += nthr) {
        const double k = vat(t.data, chain, i, 0.0), x = th[i];
        g[i] += k / x - 1.0;
        if (H) H[i * ldh + i] += k / (x * x);
      }
      break;
    case OMC_TERM_GAMMA_RESPONSE:
      for (int i = tid; i < n; i += nthr) {
        const double x = th[i];
        const double sh = vat(t.p1, chain, t.p1_len > 1 ? i : 0, 1.0), rt = vat(t.p2, chain, t.p2_len > 1 ? i : 0, 1.0);
        g[i] += (sh - 1.0) / x - rt;
        if (H) H[i * ldh + i] += (sh - 1.0) / (x * x);
      }
      break;
    case OMC_TERM_NORMAL_RESPONSE: {
      const double s = vat(t.scalar, chain, 0, 1.0);
      for (int i = tid; i < n; i += nthr) {
        double q = 0.0;
        if (t.mat_kind == OMC_MAT_DENSE) {
          for (int j = 0; j < n; ++j) {
            const double pij = mat_at(OMC_MAT_DENSE, t.P, chain, n, i, j);
            q += pij * (th[j] - vat(t.p1, chain, t.p1_len > 1 ? j : 0, 0.0));
            if (H) H[i * ldh + j] += s * pij;
          }
        } else {
          const double pii = mat_at(t.mat_kind, t.P, chain, n, i, i);
          q = pii * (th[i] - vat(t.p1, chain, t.p1_len > 1 ? i : 0, 0.0));
          if (H) H[i * ldh + i] += s * pii;
        }
        g[i] += -s * q;
      }
      break;
    }
    case OMC_TERM_LOGNORMAL_RESPONSE: {
      // grad = -(1 + Q r) / theta ; H = diag(1/theta) Q diag(1/theta) - diag((1 + Q r) / theta^2), r = log(theta) - mu
      // ref: location_scale.py:340-343 (gradient), :383-399 (Hessian)
      const double s = vat(t.scalar, chain, 0, 1.0);
      for (int i = tid; i < n; i += nthr) {
        const double ti = th[i], rci = 1.0 / ti;
        double q = 0.0;
        if (t.mat_kind == OMC_MAT_DENSE) {
          for (int j = 0; j < n; ++j) {
            const double pij = mat_at(OMC_MAT_DENSE, t.P, chain, n, i, j);
            q += pij * (log(th[j]) - vat(t.p1, chain, t.p1_len > 1 ? j : 0, 0.0));
            if (H) H[i * ldh + j] += rci * (s * pij) * (1.0 / th[j]);
          }
        } else {
          const double pii = mat_at(t.mat_kind, t.P, chain, n, i, i);
          q = pii * (log(ti) - vat(t.p1, chain, t.p1_len > 1 ? i : 0, 0.0));
          if (H) H[i * ldh + i] += rci * (s * pii) * rci;
        }
        const double one_qr = 1.0 + s * q;
        g[i] += -rci * one_qr;
        if (H) H[i * ldh + i] -= rci * rci * one_qr;
      }
      break;
    }
    case OMC_TERM_NORMAL_LINEAR: {
      const double s = vat(t.scalar, chain, 0, 1.0);
      const double* rec = t.stats.ptr + (long long)chain * t.stats.chain_stride;
      const double* G = rec;
      const double* gv = rec + n * n;
      for (int j = tid; j < n; j += nthr) {
        const double dj = t.transform_exp ? exp(th[j]) : 1.0;   // d f_j / d theta_j
        double gf = 0.0;
        for (int k = 0; k < n; ++k) {
          const double ek = t.transform_exp ? exp(th[k]) : 1.0;
          gf = fma(G[j * n + k], t.transform_exp ? ek : th[k], gf);
          if (H) H[j * ldh + k] += s * dj * G[j * n + k] * ek;
        }
        g[j] += s * dj * (gv[j] - gf);
      }
      break;
    }
    default:
      break;
  }
}

// The reference's finite differences for one term (warp-cooperative; th is a scratch copy the warp may perturb).
//   grad_k = [l(th + h/2 e_k) - l(th - h/2 e_k)] / h                       distribution.py:124-158
//   H[:,k] = [grad(th - h/2 e_k) - grad(th + h/2 e_k)] / h                 distribution.py:160-198
__device__ void term_grad_fd_warp(const omc_term_t& t, int n, int chain, double* th, double* gout /*n, lane-strided*/) {
  const int lane = threadIdx.x & 31;
  const double h = 1e-4;
  for (int k = 0; k < n; ++k) {
    const double x0 = th[k];
    __syncwarp();
    if (lane == 0) th[k] = x0 + h / 2;
    __syncwarp();
    const double lp = term_logp_warp(t, n, chain, th);
    __syncwarp();
    if (lane == 0) th[k] = x0 + (-h / 2);
    __syncwarp();
    const double lm = term_logp_warp(t, n, chain, th);
    __syncwarp();
    if (lane == 0) { th[k] = x0; gout[k] = (lp - lm) / h; }
    __syncwarp();
  }
}

// warp-cooperative gradient (+ optional Hessian) of the whole model at th (shared memory, n doubles).
// scratch: >= 3n doubles of shared memory private to the warp.
__device__ void model_grad_hess_warp(const omc_mh_model_t& m, int chain, const double* th, int method, double* g,
                                     double* H, int ldh, double* scratch) {
  const int lane = threadIdx.x & 31, n = m.n_elem;
  for (int i = lane; i < n; i += 32) g[i] = 0.0;
  if (H)   // row by row, lanes over the columns: no integer division by a run-time n
    for (int r = 0; r < n; ++r)
      for (int c = lane; c < n; c += 32) H[r * ldh + c] = 0.0;
  __syncwarp();
  for (int k = 0; k < m.n_terms; ++k) {
    const omc_term_t& t = m.terms[k];
    if (method == 0 || t.kind == OMC_TERM_NORMAL_RESPONSE || t.kind == OMC_TERM_LOGNORMAL_RESPONSE ||
        t.kind == OMC_TERM_NORMAL_LINEAR) {   // the reference differentiates these analytically too
      term_grad_hess_analytic(t, n, chain, th, g, H, ldh, lane, 32);
      __syncwarp();
      continue;
    }
    double* thw = scratch;          // perturbed copy
    double* gt = scratch + n;       // term gradient
    double* gp = scratch + 2 * n;   // gradient at a perturbed point
    for (int i = lane; i < n; i += 32) thw[i] = th[i];
    __syncwarp();
    term_grad_fd_warp(t, n, chain, thw, gt);
    for (int i = lane; i < n; i += 32) g[i] += gt[i];
    __syncwarp();
    if (H) {
      const double h = 1e-4;
      for (int c = 0; c < n; ++c) {
        const double x0 = thw[c];
        __syncwarp();
        if (lane == 0) thw[c] = x0 + h / 2;
        __syncwarp();
        term_grad_fd_warp(t, n, chain, thw, gp);
        for (int i = lane; i < n; i += 32) gt[i] = gp[i];  // gt <- grad_plus (term gradient already added to g)
        __syncwarp();
        if (lane == 0) thw[c] = x0 + (-h / 2);
        __syncwarp();
        term_grad_fd_warp(t, n, chain, thw, gp);             // gp = grad_minus
        for (int i = lane; i < n; i += 32) H[i * ldh + c] += (gp[i] - gt[i]) / h;
        __syncwarp();
        if (lane == 0) thw[c] = x0;
        __syncwarp();
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------- probes
__global__ void __launch_bounds__(MH_WARPS * 32) mh_logp_kernel(omc_mh_model_t m, const double* theta, double* out,
                                                               int accumulate) {
  extern __shared__ double sm[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int chain = blockIdx.x * MH_WARPS + warp;
  if (chain >= m.n_chains) return;
  double* th = sm + warp * m.n_elem;
  for (int i = lane; i < m.n_elem; i += 32) th[i] = theta[(long long)chain * m.n_elem + i];
  __syncwarp();
  const double lp = model_logp_warp(m, chain, th);
  if (lane == 0) out[chain] = accumulate ? out[chain] + lp : lp;
}

__global__ void __launch_bounds__(MH_WARPS * 32) mh_grad_hess_kernel(omc_mh_model_t m, const double* theta, int method,
                                                                    double* grad, double* hess) {
  extern __shared__ double sm[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, n = m.n_elem;
  const int chain = blockIdx.x * MH_WARPS + warp;
  if (chain >= m.n_chains) return;
  double* base = sm + warp * (5 * n);
  double* th = base;
  double* g = base + n;
  double* scratch = base + 2 * n;
  for (int i = lane; i < n; i += 32) th[i] = theta[(long long)chain * n + i];
  __syncwarp();
  double* H = hess ? hess + (long long)chain * n * n : nullptr;  // accumulate straight into global memory
  model_grad_hess_warp(m, chain, th, method, g, H, n, scratch);
  __syncwarp();
  for (int i = lane; i < n; i += 32) grad[(long long)chain * n + i] = g[i];
}

// ---------------------------------------------------------------------------------------------- random walk
// Contribution of element e (value x) to a term that is a SUM over elements (Poisson / Gamma / Uniform / Normal with an
// identity or diagonal precision), up to constants that do not depend on x.  Used by the column-parallel
// RandomWalkLoop: for such models the accept ratio of a column step involves only that column's elements.
__device__ __forceinline__ bool term_is_separable(const omc_term_t& t) {
  return t.kind == OMC_TERM_POISSON_RATE || t.kind == OMC_TERM_GAMMA_RESPONSE || t.kind == OMC_TERM_UNIFORM_RESPONSE ||
         (t.kind == OMC_TERM_NORMAL_RESPONSE && t.mat_kind != OMC_MAT_DENSE);
}
__device__ double term_logp_elem(const omc_term_t& t, int n, int chain, int e, double x) {
  switch (t.kind) {
    case OMC_TERM_POISSON_RATE: {
      const double k = vat(t.data, chain, e, 0.0);
      double lp = omc_xlogy(k, x) - lgamma(k + 1.0) - x;
      if (!(x >= 0.0)) lp = nan("");
      else if (!(k >= 0.0) || floor(k) != k) lp = -INFINITY;
      return lp;
    }
    case OMC_TERM_GAMMA_RESPONSE: {
      const double sh = vat(t.p1, chain, t.p1_len > 1 ? e : 0, 1.0), rt = vat(t.p2, chain, t.p2_len > 1 ? e : 0, 1.0);
      const double scale = 1.0 / rt, y = x / scale;
      double lp = omc_xlogy(sh - 1.0, y) - y - lgamma(sh) - log(scale);
      if (!(y >= 0.0)) lp = isnan(y) ? y : -INFINITY;
      return lp;
    }
    case OMC_TERM_NORMAL_RESPONSE: {
      if (x < t.dom_lo || x > t.dom_hi) return -INFINITY;
      const double r = x - vat(t.p1, chain, t.p1_len > 1 ? e : 0, 0.0);
      return -0.5 * vat(t.scalar, chain, 0, 1.0) * mat_at(t.mat_kind, t.P, chain, n, e, e) * r * r;
    }
    default:
      return 0.0;   // Uniform: constant
  }
}

__global__ void __launch_bounds__(MH_WARPS * 32) random_walk_kernel(omc_random_walk_t a) {
  extern __shared__ double sm[];
  const omc_mh_model_t& m = a.model;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, n = m.n_elem;
  const int chain = blockIdx.x * MH_WARPS + warp;
  if (chain >= m.n_chains) return;
  double* cur = sm + warp * (2 * n);
  double* prop = cur + n;
  double* gth = a.theta + (long long)chain * n;
  for (int i = lane; i < n; i += 32) cur[i] = prop[i] = gth[i];
  __syncwarp();
  const OmcRng rng = to_rng(a.rng);
  const long long sw = a.rng.sweep ? (long long)(*a.rng.sweep) : 0ll;
  const int n_steps = a.loop ? a.n_rep : 1;
  const int p_prop = a.loop ? a.p_dim : n;                 // elements proposed per step
  const unsigned blocks_per_step = (unsigned)((p_prop + 1) / 2 + 1);
  const double* dz = a.debug_z ? a.debug_z + sw * a.debug_sweep_stride_z + (long long)chain * n_steps * p_prop : nullptr;
  const double* du = a.debug_u ? a.debug_u + sw * a.debug_sweep_stride_u + (long long)chain * n_steps : nullptr;
  double logp_cur = model_logp_warp(m, chain, cur);
  long long n_acc = 0;
  bool separable = a.loop != 0;
  for (int k = 0; k < m.n_terms; ++k) separable = separable && term_is_separable(m.terms[k]);
  if (separable) {
    // ---- column-parallel RandomWalkLoop: every term is a sum over elements, so the MH step of column `stp` reads and
    //      writes that column only and log_accept = sum_rows [lp(new) - lp(old)] + lq_rev - lq_fwd; the n_rep steps are
    //      independent and run one per lane, with the very random numbers (Philox block indices) of the sequential
    //      loop.  The running total the sequential loop carries (logp_cur) is rebuilt by a prefix sum for the probes.
    for (int stp0 = 0; stp0 < n_steps; stp0 += 32) {
      const int stp = stp0 + lane;
      const bool live = stp < n_steps;
      double lq_fwd = 0.0, lq_rev = 0.0, dlp = 0.0;
      if (live) {
        for (int q = 0; q < p_prop; ++q) {
          const int row = q, col = stp, e = row * a.n_rep + col;
          const double stepv = vat(a.step, chain, (a.step_rows > 1 ? row : 0) * (a.step_cols > 1 ? a.n_rep : 1) +
                                                      (a.step_cols > 1 ? col : 0), 0.2);
          double var;
          if (dz) var = dz[(long long)stp * p_prop + q];
          else {
            uint4 b = omc_rng_block(rng, chain, stp * blocks_per_step + (unsigned)(q >> 1));
            if (a.limits) var = (q & 1) ? omc_u01(b.z, b.w) : omc_u01(b.x, b.y);
            else {
              double z0, z1;
              omc_normal2(rng, chain, stp * blocks_per_step + (unsigned)(q >> 1), z0, z1);
              var = (q & 1) ? z1 : z0;
            }
          }
          const double mu = cur[e];
          double z;
          if (a.limits) {
            const double lb = a.limits[2 * row], ub = a.limits[2 * row + 1];
            z = omc_truncated_normal_rv(mu, stepv, lb, ub, var);
            lq_fwd += omc_truncated_normal_log_pdf(z, mu, stepv, lb, ub);
            lq_rev += omc_truncated_normal_log_pdf(mu, z, stepv, lb, ub);
          } else {
            z = mu + stepv * var;
          }
          prop[e] = z;
          for (int k = 0; k < m.n_terms; ++k)
            dlp += term_logp_elem(m.terms[k], n, chain, e, z) - term_logp_elem(m.terms[k], n, chain, e, mu);
        }
      }
      double u = 0.5;
      if (live) {
        if (du) u = du[stp];
        else {
          uint4 b = omc_rng_block(rng, chain, stp * blocks_per_step + blocks_per_step - 1);
          u = omc_u01(b.x, b.y);
        }
      }
      const double log_accept = dlp + lq_rev - lq_fwd;
      const bool accept = live && (log(u) < log_accept);
      // running total before this lane's step = logp_cur + accepted increments of the lower lanes
      double inc = accept ? dlp : 0.0, pre = inc;
      for (int d = 1; d < 32; d <<= 1) {
        const double o = __shfl_up_sync(0xffffffffu, pre, d);
        if (lane >= d) pre += o;
      }
      const double before = logp_cur + (pre - inc);
      if (a.probe && live) {
        double* pr = a.probe + ((long long)chain * n_steps + stp) * 5;
        pr[0] = before; pr[1] = before + dlp; pr[2] = lq_fwd; pr[3] = lq_rev; pr[4] = accept ? 1.0 : 0.0;
      }
      if (live)
        for (int q = 0; q < p_prop; ++q) {
          const int e = q * a.n_rep + stp;
          if (accept) cur[e] = prop[e];
        }
      logp_cur += __shfl_sync(0xffffffffu, pre, 31);
      n_acc += __popc(__ballot_sync(0xffffffffu, accept));
      __syncwarp();
    }
    for (int i = lane; i < n; i += 32) gth[i] = cur[i];
    if (a.counters && lane == 0) {
      a.counters[2 * (long long)chain] += n_acc;
      a.counters[2 * (long long)chain + 1] += n_steps;
    }
    return;
  }
  for (int stp = 0; stp < n_steps; ++stp) {
    // ---- proposal for the elements of this step: element e = i*n_rep + col (loop) or e = q (joint)
    double lq_fwd = 0.0, lq_rev = 0.0;
    for (int q = lane; q < p_prop; q += 32) {
      const int row = a.loop ? q : q / a.n_rep, col = a.loop ? stp : q % a.n_rep;
      const int e = row * a.n_rep + col;
      const double stepv = vat(a.step, chain, (a.step_rows > 1 ? row : 0) * (a.step_cols > 1 ? a.n_rep : 1) +
                                                  (a.step_cols > 1 ? col : 0), 0.2);
      double var;  // N(0,1) or U(0,1) driving this element's proposal
      if (dz) var = dz[(long long)stp * p_prop + q];
      else {
        uint4 b = omc_rng_block(rng, chain, stp * blocks_per_step + (unsigned)(q >> 1));
        if (a.limits) var = (q & 1) ? omc_u01(b.z, b.w) : omc_u01(b.x, b.y);
        else {
          double z0, z1;
          omc_normal2(rng, chain, stp * blocks_per_step + (unsigned)(q >> 1), z0, z1);
          var = (q & 1) ? z1 : z0;
        }
      }
      const double mu = cur[e];
      if (a.limits) {
        const double lb = a.limits[2 * row], ub = a.limits[2 * row + 1];
        const double z = omc_truncated_normal_rv(mu, stepv, lb, ub, var);
        prop[e] = z;
        lq_fwd += omc_truncated_normal_log_pdf(z, mu, stepv, lb, ub);
        lq_rev += omc_truncated_normal_log_pdf(mu, z, stepv, lb, ub);
      } else {
        prop[e] = mu + stepv * var;
      }
    }
    lq_fwd = omc_warp_sum(lq_fwd);
    lq_rev = omc_warp_sum(lq_rev);
    __syncwarp();
    const double logp_prop = model_logp_warp(m, chain, prop);
    // ---- accept / reject (metropolis_hastings.py:155-173)
    double u;
    if (du) u = du[stp];
    else {
      uint4 b = omc_rng_block(rng, chain, stp * blocks_per_step + blocks_per_step - 1);
      u = omc_u01(b.x, b.y);
    }
    const double log_accept = logp_prop + lq_rev - (logp_cur + lq_fwd);
    const bool accept = log(u) < log_accept;
    if (a.probe && lane == 0) {
      double* pr = a.probe + ((long long)chain * n_steps + stp) * 5;
      pr[0] = logp_cur; pr[1] = logp_prop; pr[2] = lq_fwd; pr[3] = lq_rev; pr[4] = accept ? 1.0 : 0.0;
    }
    __syncwarp();
    for (int q = lane; q < p_prop; q += 32) {
      const int row = a.loop ? q : q / a.n_rep, col = a.loop ? stp : q % a.n_rep;
      const int e = row * a.n_rep + col;
      if (accept) cur[e] = prop[e];
      else prop[e] = cur[e];
    }
    if (accept) { logp_cur = logp_prop; ++n_acc; }
    __syncwarp();
  }
  for (int i = lane; i < n; i += 32) gth[i] = cur[i];
  if (a.counters && lane == 0) {
    a.counters[2 * (long long)chain] += n_acc;
    a.counters[2 * (long long)chain + 1] += n_steps;
  }
}

// ---------------------------------------------------------------------------------------------- manifold MALA
constexpr int MM_THREADS = 128;

// proposal parameters at `th`: L = chol(H / step^2) (in Hm), mu = th + 1/2 (L L')^-1 g.  Returns false if not PD / NaN.
// ref: metropolis_hastings.py:325-348
__device__ bool mmala_params(const omc_mmala_t& a, int chain, const double* th, double* Hm, int ld, double* g, double* mu,
                             double* scratch) {
  const int n = a.model.n_elem, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (warp == 0) model_grad_hess_warp(a.model, chain, th, a.method, g, Hm, ld, scratch);
  __syncthreads();
  const double inv_s2 = 1.0 / (a.step * a.step);
  bool bad = false;
  for (int e = tid; e < n * n; e += MM_THREADS) {
    const double v = Hm[(e / n) * ld + (e % n)] * inv_s2;  // precision_cr = hessian_cr / step**2
    Hm[(e / n) * ld + (e % n)] = v;
    if (isnan(v) || isinf(v)) bad = true;
  }
  for (int i = tid; i < n; i += MM_THREADS)
    if (isnan(g[i]) || isinf(g[i])) bad = true;
  if (__syncthreads_or(bad)) return false;
  if (!omc_chol_block(Hm, n, ld)) return false;
  __syncthreads();
  if (warp == 0) {
    double x0 = (lane < n) ? g[lane] : 0.0, x1 = (lane + 32 < n) ? g[lane + 32] : 0.0;
    omc_warp_solve_lower(Hm, n, ld, x0, x1);
    omc_warp_solve_lower_T(Hm, n, ld, x0, x1);
    if (lane < n) mu[lane] = th[lane] + 0.5 * x0;
    if (lane + 32 < n) mu[lane + 32] = th[lane + 32] + 0.5 * x1;
  }
  __syncthreads();
  return true;
}

// log N(x | mu, (L L')^-1) up to the constant the reference drops: sum log diag L - 1/2 |L'(x - mu)|^2
// ref: metropolis_hastings.py:350-373.  Called by warp 0 only.
__device__ double mmala_log_density_warp(const double* L, int n, int ld, const double* x, const double* mu) {
  const int lane = threadIdx.x & 31;
  const double r0 = (lane < n) ? x[lane] - mu[lane] : 0.0, r1 = (lane + 32 < n) ? x[lane + 32] - mu[lane + 32] : 0.0;
  double w0, w1;
  omc_warp_mul_lower_T(L, n, ld, r0, r1, w0, w1);
  double ld_sum = 0.0;
  if (lane < n) ld_sum += log(L[lane * ld + lane]);
  if (lane + 32 < n) ld_sum += log(L[(lane + 32) * ld + lane + 32]);
  ld_sum = omc_warp_sum(ld_sum);
  const double ww = omc_warp_sum(w0 * w0 + w1 * w1);
  return ld_sum - 0.5 * ww;
}

__global__ void __launch_bounds__(MM_THREADS) mmala_kernel(omc_mmala_t a) {
  extern __shared__ double sm[];
  const int n = a.model.n_elem, ld = n + 1, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int chain = blockIdx.x;
  double* Hm = sm;              // n x ld
  double* cur = Hm + n * ld;    // n
  double* prop = cur + n;       // n
  double* g = prop + n;         // n
  double* mu = g + n;           // n
  double* zv = mu + n;          // n
  double* scratch = zv + n;     // 3n
  __shared__ double sc[8];
  double* gth = a.theta + (long long)chain * n;
  for (int i = tid; i < n; i += MM_THREADS) cur[i] = gth[i];
  __syncthreads();
  const long long sw = a.rng.sweep ? (long long)(*a.rng.sweep) : 0ll;
  const OmcRng rng = to_rng(a.rng);
  int status = 0;
  bool ok = mmala_params(a, chain, cur, Hm, ld, g, mu, scratch);
  if (!ok) status |= OMC_STATUS_NOT_PD;
  if (ok) {
    // z, then prop = mu + L^-T z  (gmrf.sample_normal, gmrf.py:29-61)
    if (a.debug_z) {
      const double* dz = a.debug_z + sw * a.debug_sweep_stride_z + (long long)chain * n;
      for (int i = tid; i < n; i += MM_THREADS) zv[i] = dz[i];
    } else {
      for (int t = tid; 2 * t < n; t += MM_THREADS) {
        double z0, z1;
        omc_normal2(rng, chain, t, z0, z1);
        zv[2 * t] = z0;
        if (2 * t + 1 < n) zv[2 * t + 1] = z1;
      }
    }
    __syncthreads();
    if (warp == 0) {
      double x0 = (lane < n) ? zv[lane] : 0.0, x1 = (lane + 32 < n) ? zv[lane + 32] : 0.0;
      omc_warp_solve_lower_T(Hm, n, ld, x0, x1);
      if (lane < n) prop[lane] = x0 + mu[lane];
      if (lane + 32 < n) prop[lane + 32] = x1 + mu[lane + 32];
      __syncwarp();
      const double lq = mmala_log_density_warp(Hm, n, ld, prop, mu);
      const double lpc = model_logp_warp(a.model, chain, cur);
      const double lpp = model_logp_warp(a.model, chain, prop);
      if (lane == 0) { sc[0] = lpc; sc[1] = lpp; sc[2] = lq; }
    }
    __syncthreads();
    if (a.probe_mu) for (int i = tid; i < n; i += MM_THREADS) a.probe_mu[(long long)chain * n + i] = mu[i];
    if (a.probe_prop) for (int i = tid; i < n; i += MM_THREADS) a.probe_prop[(long long)chain * n + i] = prop[i];
    if (a.probe_L)
      for (int e = tid; e < n * n; e += MM_THREADS)
        a.probe_L[(long long)chain * n * n + e] = ((e % n) <= (e / n)) ? Hm[(e / n) * ld + (e % n)] : 0.0;
    __syncthreads();
    // reverse proposal parameters at the proposed point
    const bool ok2 = mmala_params(a, chain, prop, Hm, ld, g, mu, scratch);
    if (!ok2) { status |= OMC_STATUS_OUT_OF_SUPPORT; ok = false; }  // invalid PROPOSAL: reject, chain stays healthy
    else if (warp == 0) {
      const double lqr = mmala_log_density_warp(Hm, n, ld, cur, mu);
      if (lane == 0) sc[3] = lqr;
    }
    __syncthreads();
  }
  bool accept = false;
  double log_accept = nan("");
  if (ok) {
    double u;
    if (a.debug_u) u = a.debug_u[sw * a.debug_sweep_stride_u + chain];
    else {
      uint4 b = omc_rng_block(rng, chain, 0xFFFFu);
      u = omc_u01(b.x, b.y);
    }
    log_accept = sc[1] + sc[3] - (sc[0] + sc[2]);
    accept = log(u) < log_accept;
    if (isnan(log_accept)) status |= isnan(sc[0]) ? OMC_STATUS_NAN : OMC_STATUS_OUT_OF_SUPPORT;
  }
  if (accept)
    for (int i = tid; i < n; i += MM_THREADS) gth[i] = prop[i];
  if (tid == 0) {
    if (a.counters) {
      a.counters[2 * (long long)chain] += accept ? 1 : 0;
      a.counters[2 * (long long)chain + 1] += 1;
    }
    if (a.status && status) atomicOr(&a.status[chain], status);
    if (a.probe_scalars) {
      double* ps = a.probe_scalars + (long long)chain * 6;
      ps[0] = sc[0]; ps[1] = sc[1]; ps[2] = sc[2]; ps[3] = sc[3]; ps[4] = log_accept; ps[5] = accept ? 1.0 : 0.0;
    }
  }
}

// ---- warp-per-chain ManifoldMALA (n_elem <= 32): the whole step of mmala_kernel by one warp, MW_WARPS chains per CTA.
// The CTA-per-chain kernel above spends its time in __syncthreads around a 32 x 32 Cholesky that three of its four warps
// barely take part in; here nothing synchronises beyond a warp, and 4-5x as many chains are resident per SM.  Same
// operation order per element => same numbers as mmala_kernel.
constexpr int MW_WARPS = 4;

__device__ bool mmala_params_warp(const omc_mmala_t& a, int chain, const double* th, double* Hm, int ld, double* g,
                                  double* mu, double* scratch) {
  const int n = a.model.n_elem, lane = threadIdx.x & 31;
  model_grad_hess_warp(a.model, chain, th, a.method, g, Hm, ld, scratch);
  __syncwarp();
  const double inv_s2 = 1.0 / (a.step * a.step);
  bool bad = false;
  for (int r = 0; r < n; ++r)
    for (int c = lane; c < n; c += 32) {
      const double v = Hm[r * ld + c] * inv_s2;
      Hm[r * ld + c] = v;
      if (isnan(v) || isinf(v)) bad = true;
    }
  for (int i = lane; i < n; i += 32)
    if (isnan(g[i]) || isinf(g[i])) bad = true;
  __syncwarp();
  if (__any_sync(0xffffffffu, bad)) return false;
  if (!omc_chol_warp(Hm, n, ld)) return false;
  __syncwarp();
  double x0 = (lane < n) ? g[lane] : 0.0, x1 = 0.0;
  omc_warp_solve_lower(Hm, n, ld, x0, x1);
  omc_warp_solve_lower_T(Hm, n, ld, x0, x1);
  if (lane < n) mu[lane] = th[lane] + 0.5 * x0;
  __syncwarp();
  return true;
}

__global__ void __launch_bounds__(MW_WARPS * 32) mmala_warp_kernel(omc_mmala_t a) {
  extern __shared__ double sm[];
  const int n = a.model.n_elem, ld = n + 1, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int chain = blockIdx.x * MW_WARPS + warp;
  if (chain >= a.model.n_chains) return;
  double* Hm = sm + (size_t)warp * (n * ld + 8 * n);   // n x ld
  double* cur = Hm + n * ld;
  double* prop = cur + n;
  double* g = prop + n;
  double* mu = g + n;
  double* zv = mu + n;
  double* scratch = zv + n;     // 3n
  double* gth = a.theta + (long long)chain * n;
  if (lane < n) cur[lane] = gth[lane];
  __syncwarp();
  const long long sw = a.rng.sweep ? (long long)(*a.rng.sweep) : 0ll;
  const OmcRng rng = to_rng(a.rng);
  int status = 0;
  double lpc = 0.0, lpp = 0.0, lq = 0.0, lqr = 0.0;
  bool ok = mmala_params_warp(a, chain, cur, Hm, ld, g, mu, scratch);
  if (!ok) status |= OMC_STATUS_NOT_PD;
  if (ok) {
    if (a.debug_z) {
      const double* dz = a.debug_z + sw * a.debug_sweep_stride_z + (long long)chain * n;
      if (lane < n) zv[lane] = dz[lane];
    } else if (2 * lane < n) {
      double z0, z1;
      omc_normal2(rng, chain, lane, z0, z1);
      zv[2 * lane] = z0;
      if (2 * lane + 1 < n) zv[2 * lane + 1] = z1;
    }
    __syncwarp();
    double x0 = (lane < n) ? zv[lane] : 0.0, x1 = 0.0;
    omc_warp_solve_lower_T(Hm, n, ld, x0, x1);
    if (lane < n) prop[lane] = x0 + mu[lane];
    __syncwarp();
    lq = mmala_log_density_warp(Hm, n, ld, prop, mu);
    lpc = model_logp_warp(a.model, chain, cur);
    lpp = model_logp_warp(a.model, chain, prop);
    if (a.probe_mu && lane < n) a.probe_mu[(long long)chain * n + lane] = mu[lane];
    if (a.probe_prop && lane < n) a.probe_prop[(long long)chain * n + lane] = prop[lane];
    if (a.probe_L)
      for (int e = lane; e < n * n; e += 32)
        a.probe_L[(long long)chain * n * n + e] = ((e % n) <= (e / n)) ? Hm[(e / n) * ld + (e % n)] : 0.0;
    __syncwarp();
    const bool ok2 = mmala_params_warp(a, chain, prop, Hm, ld, g, mu, scratch);
    if (!ok2) { status |= OMC_STATUS_OUT_OF_SUPPORT; ok = false; }
    else lqr = mmala_log_density_warp(Hm, n, ld, cur, mu);
  }
  bool accept = false;
  double log_accept = nan("");
  if (ok) {
    double u;
    if (a.debug_u) u = a.debug_u[sw * a.debug_sweep_stride_u + chain];
    else {
      uint4 b = omc_rng_block(rng, chain, 0xFFFFu);
      u = omc_u01(b.x, b.y);
    }
    log_accept = lpp + lqr - (lpc + lq);
    accept = log(u) < log_accept;
    if (isnan(log_accept)) status |= isnan(lpc) ? OMC_STATUS_NAN : OMC_STATUS_OUT_OF_SUPPORT;
  }
  if (accept && lane < n) gth[lane] = prop[lane];
  if (lane == 0) {
    if (a.counters) {
      a.counters[2 * (long long)chain] += accept ? 1 : 0;
      a.counters[2 * (long long)chain + 1] += 1;
    }
    if (a.status && status) atomicOr(&a.status[chain], status);
    if (a.probe_scalars) {
      double* ps = a.probe_scalars + (long long)chain * 6;
      ps[0] = lpc; ps[1] = lpp; ps[2] = lq; ps[3] = lqr; ps[4] = log_accept; ps[5] = accept ? 1.0 : 0.0;
    }
  }
}

// ---- ManifoldMALA on a model whose terms are all sums over elements (Poisson rate, Gamma / Uniform response, Normal
// response with an identity or diagonal precision): the Hessian is DIAGONAL, so L = sqrt(diag), the two triangular
// solves are two divisions, and the whole step of mmala_warp_kernel is O(n) per chain with one element per lane and no
// matrix in shared memory.  Every expression is the one the dense path evaluates on that diagonal (its Cholesky of a
// diagonal matrix takes the square roots and leaves exact zeros), so the chains are the same numbers.  C4a (Poisson
// counts with a Gamma prior) is this case: 40k issued warp instructions per chain step became ~2k.
constexpr int MD_WARPS = 8;

// gradient (positive log-pdf) and Hessian diagonal (negative log-pdf) of element i at x; same expressions and the same
// accumulation order over the terms as term_grad_hess_analytic
__device__ __forceinline__ void elem_grad_hess(const omc_mh_model_t& m, int n, int chain, int i, double x, double& g,
                                               double& h) {
  g = 0.0;
  h = 0.0;
  for (int k = 0; k < m.n_terms; ++k) {
    const omc_term_t& t = m.terms[k];
    switch (t.kind) {
      case OMC_TERM_POISSON_RATE: {
        const double kk = vat(t.data, chain, i, 0.0);
        g += kk / x - 1.0;
        h += kk / (x * x);
        break;
      }
      case OMC_TERM_GAMMA_RESPONSE: {
        const double sh = vat(t.p1, chain, t.p1_len > 1 ? i : 0, 1.0), rt = vat(t.p2, chain, t.p2_len > 1 ? i : 0, 1.0);
        g += (sh - 1.0) / x - rt;
        h += (sh - 1.0) / (x * x);
        break;
      }
      case OMC_TERM_NORMAL_RESPONSE: {
        const double s = vat(t.scalar, chain, 0, 1.0);
        const double pii = mat_at(t.mat_kind, t.P, chain, n, i, i);
        const double q = pii * (x - vat(t.p1, chain, t.p1_len > 1 ? i : 0, 0.0));
        h += s * pii;
        g += -s * q;
        break;
      }
      default:
        break;   // Uniform: constant
    }
  }
}

// proposal parameters of element `lane` at x: L = sqrt(h / step^2), mu = x + 1/2 (g / L) / L; false (uniformly) when any
// element is NaN / inf or has a non-positive pivot (what mmala_params_warp reports for the dense form)
__device__ __forceinline__ bool mmala_params_diag(const omc_mmala_t& a, int n, int chain, int lane, double x, double& L,
                                                  double& mu) {
  double g = 0.0, h = 1.0;
  if (lane < n) elem_grad_hess(a.model, n, chain, lane, x, g, h);
  const double v = h * (1.0 / (a.step * a.step));
  const bool bad = (lane < n) && (isnan(v) || isinf(v) || isnan(g) || isinf(g) || !(v > 0.0));
  if (__any_sync(0xffffffffu, bad)) return false;
  L = sqrt(v);
  double x0 = g / L;
  x0 = x0 / L;
  mu = x + 0.5 * x0;
  return true;
}
__device__ __forceinline__ double mmala_log_density_diag(int n, int lane, double L, double x, double mu) {
  const double w0 = (lane < n) ? L * (x - mu) : 0.0;
  const double ld_sum = omc_warp_sum((lane < n) ? log(L) : 0.0);
  const double ww = omc_warp_sum(w0 * w0 + 0.0 * 0.0);
  return ld_sum - 0.5 * ww;
}

__global__ void __launch_bounds__(MD_WARPS * 32) mmala_diag_kernel(omc_mmala_t a) {
  extern __shared__ double sm[];
  const int n = a.model.n_elem, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int chain = blockIdx.x * MD_WARPS + warp;
  if (chain >= a.model.n_chains) return;
  double* cur = sm + (size_t)warp * 2 * n;     // model_logp_warp reads the states through memory
  double* prop = cur + n;
  double* gth = a.theta + (long long)chain * n;
  const double xc = (lane < n) ? gth[lane] : 0.0;
  if (lane < n) cur[lane] = xc;
  __syncwarp();
  const long long sw = a.rng.sweep ? (long long)(*a.rng.sweep) : 0ll;
  const OmcRng rng = to_rng(a.rng);
  int status = 0;
  double lpc = 0.0, lpp = 0.0, lq = 0.0, lqr = 0.0, L = 1.0, mu = 0.0, xp = 0.0;
  bool ok = mmala_params_diag(a, n, chain, lane, xc, L, mu);
  if (!ok) status |= OMC_STATUS_NOT_PD;
  if (ok) {
    double z = 0.0;
    if (a.debug_z) {
      if (lane < n) z = a.debug_z[sw * a.debug_sweep_stride_z + (long long)chain * n + lane];
    } else if (lane < n) {
      double z0, z1;
      omc_normal2(rng, chain, lane >> 1, z0, z1);   // pair t holds elements 2t, 2t + 1
      z = (lane & 1) ? z1 : z0;
    }
    xp = z / L + mu;
    if (lane < n) prop[lane] = xp;
    __syncwarp();
    lq = mmala_log_density_diag(n, lane, L, xp, mu);
    lpc = model_logp_warp(a.model, chain, cur);
    lpp = model_logp_warp(a.model, chain, prop);
    if (a.probe_mu && lane < n) a.probe_mu[(long long)chain * n + lane] = mu;
    if (a.probe_prop && lane < n) a.probe_prop[(long long)chain * n + lane] = xp;
    if (a.probe_L && lane < n)
      for (int c = 0; c < n; ++c) a.probe_L[(long long)chain * n * n + lane * n + c] = (c == lane) ? L : 0.0;
    double L2 = 1.0, mu2 = 0.0;
    const bool ok2 = mmala_params_diag(a, n, chain, lane, xp, L2, mu2);
    if (!ok2) { status |= OMC_STATUS_OUT_OF_SUPPORT; ok = false; }
    else lqr = mmala_log_density_diag(n, lane, L2, xc, mu2);
  }
  bool accept = false;
  double log_accept = nan("");
  if (ok) {
    double u;
    if (a.debug_u) u = a.debug_u[sw * a.debug_sweep_stride_u + chain];
    else {
      uint4 b = omc_rng_block(rng, chain, 0xFFFFu);
      u = omc_u01(b.x, b.y);
    }
    log_accept = lpp + lqr - (lpc + lq);
    accept = log(u) < log_accept;
    if (isnan(log_accept)) status |= isnan(lpc) ? OMC_STATUS_NAN : OMC_STATUS_OUT_OF_SUPPORT;
  }
  if (accept && lane < n) gth[lane] = xp;
  if (lane == 0) {
    if (a.counters) {
      a.counters[2 * (long long)chain] += accept ? 1 : 0;
      a.counters[2 * (long long)chain + 1] += 1;
    }
    if (a.status && status) atomicOr(&a.status[chain], status);
    if (a.probe_scalars) {
      double* ps = a.probe_scalars + (long long)chain * 6;
      ps[0] = lpc; ps[1] = lpp; ps[2] = lq; ps[3] = lqr; ps[4] = log_accept; ps[5] = accept ? 1.0 : 0.0;
    }
  }
}

__global__ void truncnorm_rv_kernel(const double* mean, const double* scale, const double* lower, const double* upper,
                                    const double* u, long long n, double* out) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = omc_truncated_normal_rv(mean[i], scale[i], lower[i], upper[i], u[i]);
}
__global__ void truncnorm_logpdf_kernel(const double* x, const double* mean, const double* scale, const double* lower,
                                        const double* upper, long long n, double* out) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = omc_truncated_normal_log_pdf(x[i], mean[i], scale[i], lower[i], upper[i]);
}

int check_model(const omc_mh_model_t* m, const char* who) {
  OMC_REQUIRE(m->n_chains >= 1 && m->n_elem >= 1 && m->n_terms >= 0 && m->n_terms <= 4, "%s: bad model shape", who);
  for (int k = 0; k < m->n_terms; ++k) {
    const omc_term_t& t = m->terms[k];
    OMC_REQUIRE(t.kind >= 1 && t.kind <= 6, "%s: unknown term kind %d", who, t.kind);
    if (t.kind == OMC_TERM_POISSON_RATE) OMC_REQUIRE(t.data.ptr, "%s: Poisson term without counts", who);
    if (t.kind == OMC_TERM_NORMAL_RESPONSE || t.kind == OMC_TERM_LOGNORMAL_RESPONSE)
      OMC_REQUIRE(t.mat_kind == OMC_MAT_EYE || t.P.ptr, "%s: Normal term without precision", who);
    if (t.kind == OMC_TERM_NORMAL_LINEAR)
      OMC_REQUIRE(t.stats.ptr && t.n_data >= 1 && m->n_elem <= 64, "%s: Normal-linear term needs a regression record", who);
  }
  return 0;
}

}  // namespace

extern "C" {

int omc_mh_logp_acc(const omc_mh_model_t* model, const double* theta, double* out, int accumulate, void* stream) {
  OMC_REQUIRE(model && theta && out, "omc_mh_logp: null argument");
  if (int rc = check_model(model, "omc_mh_logp")) return rc;
  const int blocks = (model->n_chains + MH_WARPS - 1) / MH_WARPS;
  const size_t smem = (size_t)MH_WARPS * model->n_elem * sizeof(double);
  mh_logp_kernel<<<blocks, MH_WARPS * 32, smem, (cudaStream_t)stream>>>(*model, theta, out, accumulate);
  OMC_LAUNCH_CHECK();
  return 0;
}
int omc_mh_logp(const omc_mh_model_t* model, const double* theta, double* out, void* stream) {
  return omc_mh_logp_acc(model, theta, out, 0, stream);
}

int omc_mh_grad_hess(const omc_mh_model_t* model, const double* theta, int method, double* grad, double* hess,
                     void* stream) {
  OMC_REQUIRE(model && theta && grad, "omc_mh_grad_hess: null argument");
  OMC_REQUIRE(method == 0 || method == 1, "omc_mh_grad_hess: method=%d", method);
  if (int rc = check_model(model, "omc_mh_grad_hess")) return rc;
  const int blocks = (model->n_chains + MH_WARPS - 1) / MH_WARPS;
  const size_t smem = (size_t)MH_WARPS * 5 * model->n_elem * sizeof(double);
  OMC_REQUIRE(smem <= 200 * 1024, "omc_mh_grad_hess: n_elem=%d too large", model->n_elem);
  OMC_CHECK_CUDA(cudaFuncSetAttribute(mh_grad_hess_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  mh_grad_hess_kernel<<<blocks, MH_WARPS * 32, smem, (cudaStream_t)stream>>>(*model, theta, method, grad, hess);
  OMC_LAUNCH_CHECK();
  return 0;
}

int omc_random_walk(const omc_random_walk_t* a, void* stream) {
  if (a) OMC_REQUIRE_SITE(a->rng, "omc_random_walk");
  OMC_REQUIRE(a && a->theta, "omc_random_walk: null argument");
  if (int rc = check_model(&a->model, "omc_random_walk")) return rc;
  OMC_REQUIRE(a->p_dim >= 1 && a->n_rep >= 1 && a->p_dim * a->n_rep == a->model.n_elem,
              "omc_random_walk: (p_dim=%d, n_rep=%d) does not match n_elem=%d", a->p_dim, a->n_rep, a->model.n_elem);
  OMC_REQUIRE((a->step_rows == 1 || a->step_rows == a->p_dim) && (a->step_cols == 1 || a->step_cols == a->n_rep),
              "omc_random_walk: step shape (%d,%d)", a->step_rows, a->step_cols);
  const int blocks = (a->model.n_chains + MH_WARPS - 1) / MH_WARPS;
  const size_t smem = (size_t)MH_WARPS * 2 * a->model.n_elem * sizeof(double);
  OMC_REQUIRE(smem <= 200 * 1024, "omc_random_walk: n_elem=%d too large", a->model.n_elem);
  OMC_CHECK_CUDA(cudaFuncSetAttribute(random_walk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  random_walk_kernel<<<blocks, MH_WARPS * 32, smem, (cudaStream_t)stream>>>(*a);
  OMC_LAUNCH_CHECK();
  return 0;
}

int omc_mmala(const omc_mmala_t* a, void* stream) {
  if (a) OMC_REQUIRE_SITE(a->rng, "omc_mmala");
  OMC_REQUIRE(a && a->theta, "omc_mmala: null argument");
  if (int rc = check_model(&a->model, "omc_mmala")) return rc;
  const int n = a->model.n_elem;
  OMC_REQUIRE(n <= 64, "omc_mmala: n_elem=%d > 64 is not supported", n);
  OMC_REQUIRE(a->step > 0.0, "omc_mmala: step=%g", a->step);
  const size_t smem = (size_t)(n * (n + 1) + 8 * n) * sizeof(double);
  bool separable = (a->method == 0);   // analytic derivatives of a model whose terms are sums over elements
  for (int k = 0; k < a->model.n_terms; ++k) {
    const omc_term_t& t = a->model.terms[k];
    separable = separable && (t.kind == OMC_TERM_POISSON_RATE || t.kind == OMC_TERM_GAMMA_RESPONSE ||
                              t.kind == OMC_TERM_UNIFORM_RESPONSE ||
                              (t.kind == OMC_TERM_NORMAL_RESPONSE && t.mat_kind != OMC_MAT_DENSE));
  }
  if (n <= 32 && separable) {   // diagonal Hessian: one element per lane, no matrix
    const size_t smem_d = (size_t)MD_WARPS * 2 * n * sizeof(double);
    mmala_diag_kernel<<<(a->model.n_chains + MD_WARPS - 1) / MD_WARPS, MD_WARPS * 32, smem_d, (cudaStream_t)stream>>>(*a);
    OMC_LAUNCH_CHECK();
    return 0;
  }
  if (n <= 32) {   // one warp per chain
    const size_t smem_w = smem * MW_WARPS;
    OMC_CHECK_CUDA(cudaFuncSetAttribute(mmala_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_w));
    mmala_warp_kernel<<<(a->model.n_chains + MW_WARPS - 1) / MW_WARPS, MW_WARPS * 32, smem_w, (cudaStream_t)stream>>>(*a);
    OMC_LAUNCH_CHECK();
    return 0;
  }
  mmala_kernel<<<a->model.n_chains, MM_THREADS, smem, (cudaStream_t)stream>>>(*a);
  OMC_LAUNCH_CHECK();
  return 0;
}

int omc_truncnorm_rv(const double* mean, const double* scale, const double* lower, const double* upper,
                     const double* u, long long n, double* out, void* stream) {
  OMC_REQUIRE(mean && scale && lower && upper && u && out && n >= 0, "omc_truncnorm_rv: bad argument");
  if (n == 0) return 0;
  truncnorm_rv_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(mean, scale, lower, upper, u, n, out);
  OMC_LAUNCH_CHECK();
  return 0;
}
int omc_truncnorm_logpdf(const double* x, const double* mean, const double* scale, const double* lower,
                         const double* upper, long long n, double* out, void* stream) {
  OMC_REQUIRE(x && mean && scale && lower && upper && out && n >= 0, "omc_truncnorm_logpdf: bad argument");
  if (n == 0) return 0;
  truncnorm_logpdf_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(x, mean, scale, lower, upper, n,
                                                                                          out);
  OMC_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
