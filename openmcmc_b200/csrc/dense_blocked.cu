// Blocked right-looking Cholesky with an FP64 tensor-core (DMMA) trailing update, one CTA per matrix.
//   * omc_nn_dense_draw for p > 32 (SURVEY.md §8 a3, a7-a10; north star: "blocked Cholesky with a DMMA trailing update"):
//       Q = lambda*P0 + tau*G, L = chol(Q), mu = L^-T L^-1 b, beta = mu + L^-T z            (gmrf.py:167-198, 29-61)
//   * omc_dense_factor: the stand-alone forms of gmrf.cholesky / cho_solve / solve / sample_normal(_canonical) and the
//       log-determinant behind multivariate_normal_pdf for a dense precision of any size up to 512
//                                                                                           (gmrf.py:414-486, 321-348)
//
// Storage: the lower triangle of the (p + n_extra) x p augmented matrix [Q ; b'] row-major with leading dimension
// LD = 16*ceil(p/16) + 4 (so that the 8 x 4 DMMA fragment reads of a warp touch every shared-memory bank exactly twice),
// in shared memory while it fits (p <= 128) and in an L2-resident global workspace above.  The right-hand side rides
// along as one more ROW, so the forward solve w = L^-1 b is done when the factorisation ends.
//
// Per panel of NB = 16 columns:
//   1. warp 0 factors the 16 x 16 diagonal block in registers (lane = row, pivots and multipliers by shuffles; the
//      reciprocal square root is MUFU.RSQ64H + two Newton steps, no division, no CTA barrier inside the panel);
//   2. one thread per row below solves its 16 panel entries against the diagonal block (forward substitution from
//      broadcast shared-memory reads) and files them in the panel buffer;
//   3. every warp updates its share of the 8 x 8 tiles of the trailing lower triangle with
//      mma.sync.m8n8k4.f64 (SASS DMMA.8x8x4): C(ti, tj) -= P(ti) P(tj)', 4 k-steps per tile.
// Three CTA barriers per panel (p/16 panels) instead of one per column.  The two backward solves (L' mu = w, L' v = z)
// run panel by panel from the bottom: a half-warp per right-hand side on the diagonal block, one thread per row above.
//
// Epilogue (re-centred sufficient statistics): with the centre record  beta_hat | c0 = X'W(y - X beta_hat) | rss0  of
// the prologue, rss(beta) = rss0 - 2 d'c0 + d'G d, d = beta - beta_hat, needs no pass over X at all and has no
// cancellation (beta_hat is the least-squares point: c0 ~ 0 and both remaining terms are non-negative).
//   ref: sampler.py:275-284 (residual.T @ P @ residual), mcmc.py:108 (log_post)
#include "../../include/omc.h"
#include "omc_common.cuh"
#include "omc_internal.h"

namespace {

#include "omc_blocked.cuh"

__device__ __forceinline__ double bvec_at(const omc_vec_t& v, int chain, int i, double dflt) {
  return v.ptr ? v.ptr[(long long)chain * v.chain_stride + i] : dflt;
}
__device__ __forceinline__ double bmat_at(int kind, const omc_vec_t& P, int chain, int p, int i, int j) {
  if (kind == OMC_MAT_DENSE) return P.ptr[(long long)chain * P.chain_stride + (long long)i * p + j];
  if (i != j) return 0.0;
  if (kind == OMC_MAT_DIAG) return P.ptr[(long long)chain * P.chain_stride + i];
  return P.ptr ? P.ptr[(long long)chain * P.chain_stride] : 1.0;
}
// rss(beta) from the centre record (see the header comment); sd = d = beta - beta_hat in shared memory.  G is symmetric:
// thread (c, row group) sums G[r][c] d_r over its rows -- consecutive threads read consecutive addresses and the loads
// of a thread are independent, so they all go out together.
__device__ void centered_rss(const omc_nn_dense_t& a, int chain, const double* __restrict__ rec,
                             const double* __restrict__ sd, double* red) {
  const int p = a.p, tid = threadIdx.x, nt = blockDim.x;
  const double* cen = a.center.ptr + (long long)chain * a.center.chain_stride;
  double acc = 0.0;
  if (p <= nt) {
    const int groups = nt / p, c = tid % p, grp = tid / p;
    if (grp < groups) {
      const int per = (p + groups - 1) / groups, r0 = grp * per, r1 = min(p, r0 + per);
      double gd = 0.0;
#pragma unroll 8
      for (int r = r0; r < r1; ++r) gd = fma(rec[(long long)r * p + c], sd[r], gd);
      acc = sd[c] * gd;
      if (grp == 0) acc = fma(-2.0 * cen[p + c], sd[c], acc);
    }
  } else {
    for (int c = tid; c < p; c += nt) {
      double gd = 0.0;
#pragma unroll 8
      for (int r = 0; r < p; ++r) gd = fma(rec[(long long)r * p + c], sd[r], gd);
      acc = fma(sd[c], gd - 2.0 * cen[p + c], acc);
    }
  }
  const double total = omc_block_sum(acc, red);
  if (tid == 0) a.rss_out[(long long)chain * a.stats.chain_stride] = cen[2 * p] + total;
}

// ---- mbarrier + bulk async copy (TMA engine, SASS UBLKCP): the rows of G go straight into the padded matrix
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra WAIT_LOOP;\n"
      "DONE:\n"
      "}\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                   (unsigned)__cvta_generic_to_shared(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"((unsigned)__cvta_generic_to_shared(bar))
               : "memory");
}

template <int NT, bool GLOBAL_A>
__global__ void __launch_bounds__(NT) nn_blocked_draw_kernel(omc_nn_dense_t a) {
  extern __shared__ __align__(16) double sm[];
  __shared__ int s_bad;
  const int p = a.p, chain = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NW = NT / 32;
  const int pp = (p + 15) & ~15;
  double* rest;
  Workspace W = carve(sm, GLOBAL_A ? a.workspace + (long long)chain * (((p + 1 + 7) & ~7) * (long long)(pp + 4)) : nullptr,
                      p, 1, &rest);
  double* X = rest;            // 2 x pp : w -> mu | z -> v
  double* sd = X + 2 * pp;     // pp : d = beta - beta_hat
  double* red = sd + pp;       // 32
  const int LD = W.LD;
  if (tid == 0) s_bad = 0;
  const double* rec = a.stats.ptr + (long long)chain * a.stats.chain_stride;
  const double tau = bvec_at(a.tau, chain, 0, 1.0);
  const double lam = bvec_at(a.lambda, chain, 0, 1.0);
  const bool solve_only = a.mode == 1;

  // ---- the lower triangle of Q = lam*P0 + tau*G (sampler.py:180-186).  Shared-memory storage with an aligned, even-p
  //      record: one elected thread sends the rows of G through the TMA engine (1-D bulk copies, row r up to its
  //      diagonal), everybody zeroes the padding meanwhile, then the rows are scaled in place.  Otherwise plain
  //      coalesced loads, row by row.
  __shared__ __align__(8) unsigned long long bar;
  const bool dense = a.prior_kind == OMC_MAT_DENSE;
  const double* P0 = dense ? a.prior_P.ptr + (long long)chain * a.prior_P.chain_stride : nullptr;
  const bool bulk = !GLOBAL_A && (p & 1) == 0 && ((((unsigned long long)rec) & 15ull) == 0);
  if (bulk) {
    if (tid == 0) {
      mbar_init(&bar, 1);
      asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
      unsigned total = 0;
      for (int r = 0; r < p; ++r) total += (unsigned)(((r + 2) & ~1) * 8);
      mbar_expect_tx(&bar, total);
      for (int r = 0; r < p; ++r)
        bulk_g2s(W.A + (long long)r * LD, rec + (long long)r * p, (unsigned)(((r + 2) & ~1) * 8), &bar);
    }
  }
  for (int e = tid; e < W.rows_pad * PLD; e += NT) W.Pn[e] = 0.0;
  for (int r = p + 1 + warp; r < W.rows_pad; r += NW)
    for (int c = lane; c < LD; c += 32) W.A[(long long)r * LD + c] = 0.0;
  if (bulk) mbar_wait(&bar, 0);
  for (int r = warp; r < p; r += NW) {
    double* arow = W.A + (long long)r * LD;
    const double* grow = rec + (long long)r * p;
    for (int c = lane; c < LD; c += 32) {
      double q = 0.0;
      if (c <= r) {
        q = tau * (bulk ? arow[c] : grow[c]);
        if (dense) q = fma(lam, P0[(long long)r * p + c], q);
        else if (c == r) q = fma(lam, bmat_at(a.prior_kind, a.prior_P, chain, p, r, r), q);
        if (c == r && solve_only) q *= 1.0 + a.ridge_rel;     // multiplicative jitter: the centre needs no exact solve
      }
      arow[c] = q;
    }
  }
  if (a.probe_Q)
    for (int e = tid; e < p * p; e += NT) {
      const int i = e / p, j = e - i * p;
      a.probe_Q[(long long)chain * p * p + e] = lam * bmat_at(a.prior_kind, a.prior_P, chain, p, i, j) + tau * rec[e];
    }
  // b = (lam*P0) mu0 + tau*g as row p; z: injected or Philox / Box-Muller (pair t = elements 2t, 2t+1)
  for (int c = tid; c < LD; c += NT) {
    double bc = 0.0;
    if (c < p) {
      double sacc;
      if (dense) {
        sacc = 0.0;
        for (int j = 0; j < p; ++j) sacc += lam * P0[(long long)c * p + j] * bvec_at(a.mu0, chain, j, 0.0);
      } else {
        sacc = lam * bmat_at(a.prior_kind, a.prior_P, chain, p, c, c) * bvec_at(a.mu0, chain, c, 0.0);
      }
      bc = sacc + tau * rec[(long long)p * p + c];
      if (a.probe_b) a.probe_b[(long long)chain * p + c] = bc;
      double zc = 0.0;
      if (!solve_only) {
        if (a.debug_z) {
          zc = a.debug_z[(a.rng.sweep ? (long long)(*a.rng.sweep) : 0ll) * a.debug_sweep_stride + (long long)chain * p + c];
        } else {
          OmcRng rg;
          rg.seed = a.rng.seed; rg.sweep = a.rng.sweep; rg.chain_offset = a.rng.chain_offset; rg.site = a.rng.site;
          double z0, z1;
          omc_normal2(rg, chain, c >> 1, z0, z1);
          zc = (c & 1) ? z1 : z0;
        }
      }
      X[pp + c] = zc;
    }
    W.A[(long long)p * LD + c] = bc;
  }
  __syncthreads();

  const bool ok = blocked_cholesky<NT>(W, p, 1, &s_bad);
  if (!ok) {
    if (solve_only) {       // the centre may be any point: fall back to the origin
      for (int c = tid; c < p; c += NT) a.beta[(long long)chain * p + c] = 0.0;
      return;
    }
    if (tid == 0 && a.status) atomicOr(&a.status[chain], OMC_STATUS_NOT_PD);
    for (int c = tid; c < p; c += NT) a.beta[(long long)chain * p + c] = nan("");
    return;
  }
  if (a.probe_L)
    for (int e = tid; e < p * p; e += NT) {
      const int i = e / p, j = e - i * p;
      a.probe_L[(long long)chain * p * p + e] = (j <= i) ? W.A[(long long)i * LD + j] : 0.0;
    }
  for (int c = tid; c < p; c += NT) X[c] = W.A[(long long)p * LD + c];     // w = L^-1 b
  __syncthreads();
  blocked_backsolve<NT>(W, p, X, pp, solve_only ? 1 : 2);
  const double* cen = a.center.ptr ? a.center.ptr + (long long)chain * a.center.chain_stride : nullptr;
  for (int c = tid; c < p; c += NT) {
    const double m = X[c];
    if (a.probe_mu) a.probe_mu[(long long)chain * p + c] = m;
    const double bnew = solve_only ? m : m + X[pp + c];
    a.beta[(long long)chain * p + c] = bnew;
    if (cen) sd[c] = bnew - cen[c];
  }
  if (cen && a.rss_out) {
    __syncthreads();
    centered_rss(a, chain, rec, sd, red);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Stand-alone dense factorisation / solves (gmrf.cholesky, cho_solve, solve(L', z), sample_normal(_canonical), log-det)
template <int NT, bool GLOBAL_A>
__global__ void __launch_bounds__(NT) dense_factor_kernel(omc_dense_factor_t a) {
  extern __shared__ __align__(16) double sm[];
  __shared__ int s_bad;
  const int n = a.n, m = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NW = NT / 32;
  const int pp = (n + 15) & ~15;
  double* rest;
  Workspace W = carve(sm, GLOBAL_A ? a.workspace + (long long)m * (((n + 1 + 7) & ~7) * (long long)(pp + 4)) : nullptr, n,
                      1, &rest);
  double* X = rest;          // 2 x pp
  double* red = X + 2 * pp;  // 32
  const int LD = W.LD;
  if (tid == 0) s_bad = 0;
  const double* Q = a.Q + (long long)m * a.Q_stride;
  const double* b = a.b ? a.b + (long long)m * n : nullptr;
  const double* z = a.z ? a.z + (long long)m * n : nullptr;
  for (int e = tid; e < W.rows_pad * PLD; e += NT) W.Pn[e] = 0.0;
  for (int r = n + 1 + warp; r < W.rows_pad; r += NW)
    for (int c = lane; c < LD; c += 32) W.A[(long long)r * LD + c] = 0.0;
  for (int r = warp; r < n; r += NW)
    for (int c = lane; c < LD; c += 32) W.A[(long long)r * LD + c] = (c <= r) ? Q[(long long)r * n + c] : 0.0;
  for (int c = tid; c < LD; c += NT) {
    W.A[(long long)n * LD + c] = (c < n && b) ? b[c] : 0.0;
    if (c < n) X[pp + c] = z ? z[c] : 0.0;
  }
  __syncthreads();
  bool ok = true;
  if (a.factored) {        // Q already holds a lower Cholesky factor: only 1/L_jj and the forward solve are needed
    for (int j = tid; j < n; j += NT) W.sinv[j] = 1.0 / W.A[(long long)j * LD + j];
    __syncthreads();
    if (b) {               // w = L^-1 b, one column at a time (setup-time path, not a sweep kernel)
      for (int j = 0; j < n; ++j) {
        if (tid == 0) W.A[(long long)n * LD + j] *= W.sinv[j];
        __syncthreads();
        const double wj = W.A[(long long)n * LD + j];
        for (int c = j + 1 + tid; c < n; c += NT) W.A[(long long)n * LD + c] -= W.A[(long long)c * LD + j] * wj;
        __syncthreads();
      }
    }
  } else {
    ok = blocked_cholesky<NT>(W, n, 1, &s_bad);
  }
  if (!ok) {
    if (tid == 0 && a.status) atomicOr(&a.status[m], OMC_STATUS_NOT_PD);
    if (a.logdet && tid == 0) a.logdet[m] = nan("");
    for (int c = tid; c < n; c += NT) {
      if (a.x) a.x[(long long)m * n + c] = nan("");
      if (a.mean) a.mean[(long long)m * n + c] = nan("");
    }
    return;
  }
  if (a.L)
    for (int e = tid; e < n * n; e += NT) {
      const int i = e / n, j = e - i * n;
      a.L[(long long)m * n * n + e] = (j <= i) ? W.A[(long long)i * LD + j] : 0.0;
    }
  if (a.logdet) {          // log|Q| = 2 sum log L_jj
    double acc = 0.0;
    for (int j = tid; j < n; j += NT) acc += log(W.A[(long long)j * LD + j]);
    acc = omc_block_sum(acc, red);
    if (tid == 0) a.logdet[m] = 2.0 * acc;
  }
  if (!a.x && !a.mean) return;
  if (a.backward_only == 2) {   // forward solve only: mean = L^-1 b
    for (int c = tid; c < n; c += NT) {
      const double wv = W.A[(long long)n * LD + c];
      if (a.mean) a.mean[(long long)m * n + c] = wv;
      if (a.x) a.x[(long long)m * n + c] = wv + X[pp + c];
    }
    return;
  }
  // X[0] = forward-solved b (cho_solve) or b itself (backward_only: solve(L', b));  X[1] = z
  for (int c = tid; c < n; c += NT) X[c] = (a.backward_only == 1 && b) ? b[c] : W.A[(long long)n * LD + c];
  __syncthreads();
  blocked_backsolve<NT>(W, n, X, pp, 2);
  for (int c = tid; c < n; c += NT) {
    if (a.mean) a.mean[(long long)m * n + c] = X[c];
    if (a.x) a.x[(long long)m * n + c] = X[c] + X[pp + c];
  }
}

size_t smem_bytes(int p, bool global_A) {
  const int pp = (p + 15) & ~15, LD = pp + 4, rows_pad = (p + 1 + 7) & ~7;
  size_t d = (size_t)rows_pad * PLD + NB * SDLD + 3 + pp /*sinv*/ + 3 * (size_t)pp + 32;
  if (!global_A) d += (size_t)rows_pad * LD;
  return d * sizeof(double);
}

}  // namespace

long long omc_blocked_workspace_doubles(int p) {
  const int pp = (p + 15) & ~15;
  if (smem_bytes(p, false) <= 200 * 1024) return 0;
  return (long long)((p + 1 + 7) & ~7) * (pp + 4);
}

int omc_launch_blocked_draw(const omc_nn_dense_t& a, cudaStream_t st) {
  const int p = a.p;
  OMC_REQUIRE(p <= 512, "omc_nn_dense_draw: p=%d > 512 is not supported", p);
  const bool global_A = omc_blocked_workspace_doubles(p) > 0;
  OMC_REQUIRE(!global_A || a.workspace, "omc_nn_dense_draw: p=%d needs a workspace of omc_nn_dense_workspace() doubles", p);
  const size_t smem = smem_bytes(p, global_A);
  if (global_A) {
    OMC_CHECK_CUDA(cudaFuncSetAttribute(nn_blocked_draw_kernel<256, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    nn_blocked_draw_kernel<256, true><<<a.n_chains, 256, smem, st>>>(a);
  } else if (p <= 64) {
    OMC_CHECK_CUDA(cudaFuncSetAttribute(nn_blocked_draw_kernel<128, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    nn_blocked_draw_kernel<128, false><<<a.n_chains, 128, smem, st>>>(a);
  } else {
    OMC_CHECK_CUDA(cudaFuncSetAttribute(nn_blocked_draw_kernel<256, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    nn_blocked_draw_kernel<256, false><<<a.n_chains, 256, smem, st>>>(a);
  }
  OMC_LAUNCH_CHECK();
  return 0;
}

extern "C" int omc_nn_dense_workspace(int n_chains, int p, long long* doubles) {
  OMC_REQUIRE(doubles && n_chains >= 1 && p >= 1, "omc_nn_dense_workspace: bad argument");
  *doubles = omc_blocked_workspace_doubles(p) * n_chains;
  return 0;
}

extern "C" int omc_dense_factor(const omc_dense_factor_t* a, void* stream) {
  OMC_REQUIRE(a && a->Q && a->n_mats >= 1 && a->n >= 1, "omc_dense_factor: bad argument");
  OMC_REQUIRE(a->n <= 512, "omc_dense_factor: n=%d > 512 is not supported", a->n);
  const bool global_A = omc_blocked_workspace_doubles(a->n) > 0;
  OMC_REQUIRE(!global_A || a->workspace, "omc_dense_factor: n=%d needs a workspace of omc_nn_dense_workspace() doubles", a->n);
  const size_t smem = smem_bytes(a->n, global_A);
  cudaStream_t st = (cudaStream_t)stream;
  if (global_A) {
    OMC_CHECK_CUDA(cudaFuncSetAttribute(dense_factor_kernel<256, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dense_factor_kernel<256, true><<<a->n_mats, 256, smem, st>>>(*a);
  } else {
    OMC_CHECK_CUDA(cudaFuncSetAttribute(dense_factor_kernel<256, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dense_factor_kernel<256, false><<<a->n_mats, 256, smem, st>>>(*a);
  }
  OMC_LAUNCH_CHECK();
  return 0;
}
