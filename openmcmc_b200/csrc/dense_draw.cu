// Small per-chain kernels of the conjugate Gibbs updates (SURVEY.md §8 a3, a7-a10, a12):
//   omc_nn_dense_draw : Q = lambda*P0 + tau*G, Cholesky, posterior mean, MVN draw  (Rue & Held Alg. 2.5)
//   omc_quadform      : (x-mu)' P (x-mu) and #(diag P > 0)
//   omc_ng_draw       : Gamma(a0 + cnt/2, b0 + ss/2) draw
// p <= 32: one thread per COLUMN of Q with the column in registers (nn_dense_draw_kernel below); above that the blocked
// Cholesky with the DMMA trailing update of dense_blocked.cu.  One thread per chain for the scalar Gamma draw.  With the
// re-centred statistics (omc_nn_dense_t.center) the draw also leaves rss(beta) in the record, so a steady-state C2
// sweep is these latency-bound kernels alone: no pass over X.
#include "../../include/omc.h"
#include "omc_common.cuh"
#include "omc_internal.h"
#include "omc_special.cuh"

namespace {

constexpr int DD_THREADS = 256;
constexpr int PMAX = 512;
// above this p the left-looking warp kernel (14 chains per SM) runs instead of the register one (8): measured faster at
// p = 48, 56, 63 and 64 with 4096 chains (profiles/r03_draw_only.txt)
constexpr int LEFT_MIN_P = 40;

__device__ __forceinline__ double vec_at(const omc_vec_t& v, int chain, int i, double dflt) {
  return v.ptr ? v.ptr[(long long)chain * v.chain_stride + i] : dflt;
}
__device__ __forceinline__ OmcRng to_rng(const omc_rng_t& r) {
  OmcRng o;
  o.seed = r.seed; o.sweep = r.sweep; o.chain_offset = r.chain_offset; o.site = r.site;
  return o;
}

// P0[i][j] for the three storage kinds
__device__ __forceinline__ double mat_at(int kind, const omc_vec_t& P, int chain, int p, int i, int j) {
  if (kind == OMC_MAT_DENSE) return P.ptr[(long long)chain * P.chain_stride + (long long)i * p + j];
  if (i != j) return 0.0;
  if (kind == OMC_MAT_DIAG) return P.ptr[(long long)chain * P.chain_stride + i];
  return P.ptr ? P.ptr[(long long)chain * P.chain_stride] : 1.0;
}

__global__ void __launch_bounds__(DD_THREADS) nn_truncated_scan_kernel(omc_nn_dense_t a) {
  extern __shared__ double sm[];
  const int p = a.p, ld = p + 1;
  double* Q = sm;                 // p x ld, becomes L (lower triangle)
  double* b = Q + p * ld;         // p : rhs -> w -> mu
  double* z = b + p;              // p : z -> v
  double* mu0 = z + p;            // p
  double* invd = mu0 + p;         // p : 1 / L_jj
  __shared__ int bad;
  const int chain = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = DD_THREADS / 32;
  if (tid == 0) bad = 0;

  const double* rec = a.stats.ptr + (long long)chain * a.stats.chain_stride;
  const double tau = vec_at(a.tau, chain, 0, 1.0);
  const double lam = vec_at(a.lambda, chain, 0, 1.0);

  for (int i = tid; i < p; i += DD_THREADS) mu0[i] = vec_at(a.mu0, chain, i, 0.0);
  // Q = lam*P0 + tau*G  (full symmetric; reference adds the scaled prior then the likelihood Hessian, sampler.py:180-186)
  for (int e = tid; e < p * p; e += DD_THREADS) {
    int i = e / p, j = e - i * p;
    double q = lam * mat_at(a.prior_kind, a.prior_P, chain, p, i, j) + tau * rec[e];
    Q[i * ld + j] = q;
    if (a.probe_Q) a.probe_Q[(long long)chain * p * p + e] = q;
  }
  __syncthreads();
  // b = (lam*P0) mu0 + tau*g
  for (int i = tid; i < p; i += DD_THREADS) {
    double s = 0.0;
    if (a.prior_kind == OMC_MAT_DENSE) {
      for (int j = 0; j < p; ++j) s += lam * mat_at(OMC_MAT_DENSE, a.prior_P, chain, p, i, j) * mu0[j];
    } else {
      s = lam * mat_at(a.prior_kind, a.prior_P, chain, p, i, i) * mu0[i];
    }
    s += tau * rec[p * p + i];
    b[i] = s;
    if (a.probe_b) a.probe_b[(long long)chain * p + i] = s;
  }
  {
    // ---- truncated prior: one coordinate-wise Gibbs scan from the current beta (gmrf.py:201-266), warp 0
    __syncthreads();
    if (warp == 0) {
      double* bt = a.beta + (long long)chain * p;
      double x0 = (lane < p) ? bt[lane] : 0.0, x1 = (lane + 32 < p) ? bt[lane + 32] : 0.0;
      const double* du = a.debug_u
                             ? a.debug_u + (a.rng.sweep ? (long long)(*a.rng.sweep) : 0ll) * a.debug_sweep_stride +
                                   (long long)chain * p
                             : nullptr;
      OmcRng rng = to_rng(a.rng);
      for (int i = 0; i < p; ++i) {
        double part = 0.0;
        if (lane < p) part = Q[i * ld + lane] * x0;
        if (lane + 32 < p) part = fma(Q[i * ld + lane + 32], x1, part);
        const double dot = omc_warp_sum(part);
        const double xi = __shfl_sync(0xffffffffu, (i < 32) ? x0 : x1, i & 31);
        const double qii = Q[i * ld + i];
        const double v = 1.0 / qii;
        const double mean = (p == 1) ? b[0] / qii : v * (b[i] - dot + qii * xi);
        const double lo = a.trunc_lo.ptr ? vec_at(a.trunc_lo, chain, a.trunc_lo_len > 1 ? i : 0, 0.0) : -INFINITY;
        const double hi = a.trunc_hi.ptr ? vec_at(a.trunc_hi, chain, a.trunc_hi_len > 1 ? i : 0, 0.0) : INFINITY;
        double u;
        if (du) u = du[i];
        else {
          const uint4 blk = omc_rng_block(rng, chain, (unsigned int)i);
          u = omc_u01(blk.x, blk.y);
        }
        const double xn = omc_truncated_normal_rv(mean, sqrt(v), lo, hi, u);
        if (!(qii > 0.0) && lane == 0) bad = 1;
        if (lane == (i & 31)) { if (i < 32) x0 = xn; else x1 = xn; }
      }
      if (lane < p) bt[lane] = x0;
      if (lane + 32 < p) bt[lane + 32] = x1;
      if (lane == 0 && bad && a.status) atomicOr(&a.status[chain], OMC_STATUS_NOT_PD);
    }
  }
}

// ---- NormalNormal draw, dense p x p posterior precision: one thread per COLUMN, the column in registers.
// Thread c owns Q[i][c], i >= c (the lower triangle is all the reference's Cholesky reads).  Right-looking Cholesky:
// at step j thread j scales its column by 1/sqrt(Q_jj) and publishes it in shared memory (column-major L, which the
// triangular solves read afterwards); the other threads read it back as broadcasts and update their own column with
// statically indexed registers (the loop over rows is unrolled, the loop over j is not).  The right-hand side b rides
// along as one more row, so w = L^-1 b is there when the factorisation ends (ONE barrier per column, none in the solves).
// Two warps then run the backward solves L' mu = w and L' v = z (lane = row, shuffle broadcast of the pivot element).
// The previous CTA-wide kernel (256 threads, matrix in shared memory, 3 barriers per column) took 0.66 ms for the
// 4096 chains of C2, a fifth of the sweep once the pass over X became a pure stream.
template <int PR>
__global__ void __launch_bounds__((PR < 32 ? 32 : PR), (PR == 32 ? 10 : 16)) nn_dense_draw_kernel(omc_nn_dense_t a) {
  constexpr int NT = PR < 32 ? 32 : PR;
  constexpr int LD = PR + 2;                 // column stride (doubles): 16-byte aligned columns
  extern __shared__ __align__(16) double sm[];
  double* sL = sm;                           // sL[j * LD + i] = L[i][j], i >= j
  double* sw = sL + PR * LD;                 // b -> w = L^-1 b -> mu
  double* sz = sw + PR;                      // z -> v = L^-T z
  double* sinv = sz + PR;                    // 1 / L_jj
  double* sraw = sinv + PR;                  // 2 x PR: the unscaled column of the current step (double-buffered)
  __shared__ int s_bad;
  const int chain = blockIdx.x, c = threadIdx.x, lane = c & 31, warp = c >> 5, p = a.p;
  const bool live = c < p;
  if (c == 0) s_bad = 0;
  const double* rec = a.stats.ptr + (long long)chain * a.stats.chain_stride;
  const double tau = vec_at(a.tau, chain, 0, 1.0);
  const double lam = vec_at(a.lambda, chain, 0, 1.0);

  // ---- column c of Q = lam*P0 + tau*G (sampler.py:180-186), consecutive threads read consecutive addresses.  The
  //      loads are kept free of stores (a probe store between them would order every load behind the previous one).
  double col[PR];
  double diag = 0.0, bc = 0.0;
  {
    const double* gcol = rec + c;             // G[i][c] at gcol[i * p]
    const bool dense = a.prior_kind == OMC_MAT_DENSE;
    const double* pcol = dense ? a.prior_P.ptr + (long long)chain * a.prior_P.chain_stride + c : gcol;
    const double lam_d = dense ? lam : 0.0;   // one loop for the three prior kinds: the off-diagonal prior term is
#pragma unroll                                // lam * P0[i][c] for a dense prior and nothing otherwise
    for (int i = 0; i < PR; ++i) {
      double q = 0.0;
      if (live && i < p && i > c) q = fma(lam_d, pcol[i * p], tau * gcol[i * p]);
      col[i] = q;
    }
    if (live) diag = lam * mat_at(a.prior_kind, a.prior_P, chain, p, c, c) + tau * gcol[c * p];
    if (a.mode == 1) diag *= 1.0 + a.ridge_rel;
  }
  if (a.probe_Q && live) {
    for (int i = 0; i < p; ++i)
      a.probe_Q[(long long)chain * p * p + i * p + c] =
          lam * mat_at(a.prior_kind, a.prior_P, chain, p, i, c) + tau * rec[i * p + c];
  }
  if (live) {   // b = (lam*P0) mu0 + tau*g
    double sacc = 0.0;
    if (a.prior_kind == OMC_MAT_DENSE) {
      for (int j = 0; j < p; ++j) sacc += lam * mat_at(OMC_MAT_DENSE, a.prior_P, chain, p, c, j) * vec_at(a.mu0, chain, j, 0.0);
    } else {
      sacc = lam * mat_at(a.prior_kind, a.prior_P, chain, p, c, c) * vec_at(a.mu0, chain, c, 0.0);
    }
    bc = sacc + tau * rec[p * p + c];
    if (a.probe_b) a.probe_b[(long long)chain * p + c] = bc;
    // z: injected or Philox / Box-Muller (pair t = elements 2t, 2t+1; both threads of a pair draw it)
    double zc;
    if (a.mode == 1) {
      zc = 0.0;
    } else if (a.debug_z) {
      zc = a.debug_z[(a.rng.sweep ? (long long)(*a.rng.sweep) : 0ll) * a.debug_sweep_stride + (long long)chain * p + c];
    } else {
      double z0, z1;
      omc_normal2(to_rng(a.rng), chain, c >> 1, z0, z1);
      zc = (c & 1) ? z1 : z0;
    }
    sz[c] = zc;
  }

  // ---- right-looking Cholesky with the forward solve riding along.  Thread j publishes its column UNSCALED together
  //      with rd = 1/sqrt(Q_jj) (its serial section is a reciprocal square root and 32 stores); thread i > j scales its
  //      own entry L[i][j] = Q[i][j] * rd, stores it for the solves, and updates its column with the factor
  //      L[i][j] * rd.  The raw column is double-buffered, so ONE barrier per step is enough.  Pairs of rows that are
  //      dead for the whole warp (i <= j, or above the warp's first column) are skipped with a warp-uniform branch.
  const int warp_lo = warp * 32;
  for (int j = 0; j < p; ++j) {
    double* colj = sraw + (j & 1) * PR;
    if (c == j) {
      if (!(diag > 0.0)) s_bad = j + 1;      // step-stamped: a fast thread of step j + 1 cannot end step j early
      double rd;
      asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(rd) : "d"(diag));
      const double hd = 0.5 * diag;
      double e = fma(-hd, rd * rd, 0.5);
      rd = fma(rd, e, rd);
      e = fma(-hd, rd * rd, 0.5);
      rd = fma(rd, e, rd);                   // 1/sqrt(Q_jj), relative error ~1e-16
#pragma unroll
      for (int i = 0; i < PR; i += 2)          // all of it (rows <= j are never read): no branches in the serial section
        *reinterpret_cast<double2*>(colj + i) = make_double2(col[i], col[i + 1]);
      sL[j * LD + j] = diag * rd;            // L_jj
      sinv[j] = rd;
      sw[j] = bc * rd;                       // w_j
    }
    __syncthreads();
    {
      const int sb = s_bad;
      if (sb != 0 && sb <= j + 1) break;     // uniform: every thread sees the stamp of step j after the barrier
    }
    if (c > j && live) {
      const double rd = sinv[j];
      const double lc = colj[c] * rd;        // L[c][j]
      const double f = lc * rd;
      sL[j * LD + c] = lc;
      diag = fma(-lc, lc, diag);
      bc = fma(-lc, sw[j], bc);
      const int lo = max(j, warp_lo);
#pragma unroll
      for (int i0 = 0; i0 < PR; i0 += 16) {   // chunks of 16 rows: the loads of a chunk go out together
        if (i0 + 15 > lo) {                   // warp-uniform
          double2 v[8];
#pragma unroll
          for (int k = 0; k < 8; ++k) v[k] = *reinterpret_cast<const double2*>(colj + i0 + 2 * k);
#pragma unroll
          for (int k = 0; k < 8; ++k) {         // rows <= c of a live chunk are updated too: they are never read
            const int i = i0 + 2 * k;
            col[i] = fma(-v[k].x, f, col[i]);
            col[i + 1] = fma(-v[k].y, f, col[i + 1]);
          }
        }
      }
    }
  }
  __syncthreads();
  if (s_bad) {
    if (a.mode == 1) {      // the centre of the re-centred statistics may be any point: fall back to the origin
      if (live) a.beta[(long long)chain * p + c] = 0.0;
      return;
    }
    if (c == 0 && a.status) atomicOr(&a.status[chain], OMC_STATUS_NOT_PD);
    if (live) a.beta[(long long)chain * p + c] = nan("");
    return;
  }
  if (a.probe_L) {
    for (int e = c; e < p * p; e += NT) {
      const int i = e / p, j = e - i * p;
      a.probe_L[(long long)chain * p * p + e] = (j <= i) ? sL[j * LD + i] : 0.0;
    }
  }
  // ---- backward solves with L' (uses row j of L): warp 0: L' mu = w ; the last warp: L' v = z ; lane owns rows
  //      lane and lane + 32
  auto backsolve = [&](double* x) {
    double x0 = (lane < p) ? x[lane] : 0.0, x1 = (lane + 32 < p) ? x[lane + 32] : 0.0;
    for (int j = p - 1; j >= 0; --j) {
      const double xj = __shfl_sync(0xffffffffu, (j < 32) ? x0 : x1, j & 31) * sinv[j];
      if (lane == (j & 31)) { if (j < 32) x0 = xj; else x1 = xj; }
      if (lane < j) x0 = fma(-sL[lane * LD + j], xj, x0);
      if (lane + 32 < j) x1 = fma(-sL[(lane + 32) * LD + j], xj, x1);
    }
    if (lane < p) x[lane] = x0;
    if (lane + 32 < p) x[lane + 32] = x1;
  };
  if (warp == 0) backsolve(sw);
  if (warp == NT / 32 - 1) backsolve(sz);
  __syncthreads();
  const double* cen = a.center.ptr ? a.center.ptr + (long long)chain * a.center.chain_stride : nullptr;
  if (live) {
    const double m = sw[c];
    if (a.probe_mu) a.probe_mu[(long long)chain * p + c] = m;
    const double bnew = a.mode == 1 ? m : m + sz[c];
    a.beta[(long long)chain * p + c] = bnew;
    if (cen) sraw[c] = bnew - cen[c];
  }
  if (cen && a.rss_out) {
    // rss(beta) = rss0 - 2 d'c0 + d'G d from the centre record (omc.h); G is symmetric: (G d)_c from coalesced rows
    __syncthreads();
    double acc = 0.0;
    if (live) {
      double gd = 0.0;
      for (int r = 0; r < p; ++r) gd = fma(rec[r * p + c], sraw[r], gd);
      acc = sraw[c] * (gd - 2.0 * cen[p + c]);
    }
    const double total = omc_block_sum(acc, sraw + PR);
    if (c == 0) a.rss_out[(long long)chain * a.stats.chain_stride] = cen[2 * p] + total;
  }
}

template <int PR>
int launch_dense_draw(const omc_nn_dense_t& a, cudaStream_t st) {
  constexpr int NT = PR < 32 ? 32 : PR;
  const size_t smem = (size_t)(PR * (PR + 2) + 5 * PR + 32) * sizeof(double);
  nn_dense_draw_kernel<PR><<<a.n_chains, NT, smem, st>>>(a);
  OMC_LAUNCH_CHECK();
  return 0;
}

__global__ void quadform_kernel(omc_quadform_t a) {
  // one warp per chain
  const int chain = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (chain >= a.n_chains) return;
  const int p = a.p;
  double ss = 0.0, cnt = 0.0;
  if (a.kind == OMC_MAT_DENSE) {
    for (int i = lane; i < p; i += 32) {
      const double ri = vec_at(a.x, chain, i, 0.0) - vec_at(a.mu, chain, i, 0.0);
      double s = 0.0;
      for (int j = 0; j < p; ++j)
        s += mat_at(OMC_MAT_DENSE, a.P, chain, p, i, j) * (vec_at(a.x, chain, j, 0.0) - vec_at(a.mu, chain, j, 0.0));
      ss += ri * s;
      cnt += (mat_at(OMC_MAT_DENSE, a.P, chain, p, i, i) > 0.0) ? 1.0 : 0.0;
    }
  } else {
    for (int i = lane; i < p; i += 32) {
      const double ri = vec_at(a.x, chain, i, 0.0) - vec_at(a.mu, chain, i, 0.0);
      const double d = mat_at(a.kind, a.P, chain, p, i, i);
      ss += d * ri * ri;
      cnt += (d > 0.0) ? 1.0 : 0.0;
    }
  }
  ss = omc_warp_sum(ss);
  cnt = omc_warp_sum(cnt);
  if (lane == 0) {
    a.ss[chain] = ss;
    a.cnt[chain] = cnt;
  }
}

__global__ void ng_draw_kernel(omc_ng_draw_t a) {
  const int ne = a.n_elem > 0 ? a.n_elem : 1;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)a.n_chains * ne) return;
  const int chain = (int)(t / ne), k = (int)(t - (long long)chain * ne);
  const double shape = vec_at(a.a0, chain, a.a0_len > 1 ? k : 0, 0.0) + 0.5 * vec_at(a.cnt, chain, k * a.cnt_stride, 0.0);
  const double rate = vec_at(a.b0, chain, a.b0_len > 1 ? k : 0, 0.0) + 0.5 * vec_at(a.ss, chain, k * a.ss_stride, 0.0);
  if (a.probe_a) a.probe_a[t] = shape;
  if (a.probe_b) a.probe_b[t] = rate;
  double gvar;
  if (a.debug_g) gvar = a.debug_g[(a.rng.sweep ? (long long)(*a.rng.sweep) : 0ll) * a.debug_sweep_stride + t];
  else gvar = omc_std_gamma(to_rng(a.rng), chain, (unsigned int)k << 12, shape);   // 4096 Philox blocks per element
  // reference: scale = inf when rate == 0 (sampler.py:285-286)
  a.out[t] = (rate == 0.0) ? INFINITY : gvar * (1.0 / rate);
}

}  // namespace

extern "C" int omc_nn_dense_draw(const omc_nn_dense_t* args, void* stream) {
  if (args) OMC_REQUIRE_SITE(args->rng, "omc_nn_dense_draw");
  OMC_REQUIRE(args && args->stats.ptr && args->beta, "omc_nn_dense_draw: null argument");
  OMC_REQUIRE(args->p >= 1 && args->p <= PMAX, "omc_nn_dense_draw: p=%d outside [1,%d]", args->p, PMAX);
  OMC_REQUIRE(args->n_chains >= 1, "omc_nn_dense_draw: n_chains=%d", args->n_chains);
  OMC_REQUIRE(args->prior_kind >= 0 && args->prior_kind <= 2, "omc_nn_dense_draw: prior_kind=%d", args->prior_kind);
  OMC_REQUIRE(args->prior_kind == OMC_MAT_EYE || args->prior_P.ptr, "omc_nn_dense_draw: prior_P missing");
  const int p = args->p;
  if (args->truncated) {
    // p <= 64: Q in shared memory, the scan in one warp of a CTA per chain; above: one warp per chain streaming the rows
    // of G (and P0) through shared memory (trunc_scan.cu)
    if (p > 64) return omc_launch_trunc_stream(*args, (cudaStream_t)stream);
    const size_t smem = (size_t)(p * (p + 1) + 4 * p) * sizeof(double);
    OMC_CHECK_CUDA(cudaFuncSetAttribute(nn_truncated_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    nn_truncated_scan_kernel<<<args->n_chains, DD_THREADS, smem, (cudaStream_t)stream>>>(*args);
    OMC_LAUNCH_CHECK();
    return 0;
  }
  // p <= 64 without probes: one warp per chain (dense_warp.cu), the left-looking kernel with the factor in shared
  // memory above LEFT_MIN_P, Q in registers below.  Probes (Q, b, L, mu of the parity tests) go through the kernels
  // that keep the factor addressable: one thread per column (p <= 32) or the blocked Cholesky (dense_blocked.cu), which
  // also serves 64 < p <= 512.
  const bool probes = args->probe_Q || args->probe_b || args->probe_L || args->probe_mu;
  if (p <= 64 && !probes) {
    if (p > LEFT_MIN_P) return omc_launch_left_draw(*args, (cudaStream_t)stream);
    return omc_launch_warp_draw(*args, (cudaStream_t)stream);
  }
  if (p <= 8) return launch_dense_draw<8>(*args, (cudaStream_t)stream);
  if (p <= 16) return launch_dense_draw<16>(*args, (cudaStream_t)stream);
  if (p <= 32) return launch_dense_draw<32>(*args, (cudaStream_t)stream);
  return omc_launch_blocked_draw(*args, (cudaStream_t)stream);
}

extern "C" int omc_quadform(const omc_quadform_t* args, void* stream) {
  OMC_REQUIRE(args && args->x.ptr && args->ss && args->cnt, "omc_quadform: null argument");
  OMC_REQUIRE(args->kind >= 0 && args->kind <= 2, "omc_quadform: kind=%d", args->kind);
  OMC_REQUIRE(args->kind == OMC_MAT_EYE || args->P.ptr, "omc_quadform: P missing");
  const int threads = 128;
  const long long total = (long long)args->n_chains * 32;
  quadform_kernel<<<(unsigned)((total + threads - 1) / threads), threads, 0, (cudaStream_t)stream>>>(*args);
  OMC_LAUNCH_CHECK();
  return 0;
}

extern "C" int omc_ng_draw(const omc_ng_draw_t* args, void* stream) {
  if (args) OMC_REQUIRE_SITE(args->rng, "omc_ng_draw");
  OMC_REQUIRE(args && args->out, "omc_ng_draw: null argument");
  const int threads = 128;
  const long long total = (long long)args->n_chains * (args->n_elem > 0 ? args->n_elem : 1);
  ng_draw_kernel<<<(unsigned)((total + threads - 1) / threads), threads, 0, (cudaStream_t)stream>>>(*args);
  OMC_LAUNCH_CHECK();
  return 0;
}
