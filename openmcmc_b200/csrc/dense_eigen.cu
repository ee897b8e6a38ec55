// omc_nn_eigen_prep / omc_nn_eigen_draw: the dense NormalNormal draw at p <= 64 in a fixed eigenbasis.
//
// When G, g, P0 (scaled identity or positive diagonal), mu0 and the centre record are data, so is the generalized
// eigenbasis of (G, P0):  M'P0M = I, M'GM = D.  With S = lam I + tau D the posterior precision is Q = M^-T S M^-1, so
//   beta = M u,  u = S^-1 (tau h + lam m) + S^-1/2 z,  h = M'g, m = M'P0 mu0          (M S^-1/2 is a square root of Q^-1)
//   rss(beta) = rss0 - 2 e'k + e'D e,  e = u - u_hat, u_hat = M'P0 beta_hat, k = M'c0  (omc.h, the centre record)
// and a sweep's draw is an O(p) element-wise step plus one p x p mat-vec per chain: a read stream with no dependent
// chain, where the Cholesky of Q is 64 dependent pivot stages (dense_warp.cu).
//
// Prep (once per run, one CTA per chain): G~ = R^-1 G R^-1, R = diag(sqrt(P0)), in shared memory; two-sided cyclic
// Jacobi with the parallel round-robin ordering (p/2 disjoint rotations per round, one idle index for odd p) and
// Rutishauser's rotation, W accumulated; each round updates every 2 x 2 block of G~ in one step (J_k' B J_l), the
// diagonal blocks set exactly (a_pp - t a_pq, a_qq + t a_pq, 0).  A pair rotates while |a_pq| > eps sqrt|a_pp a_qq|
// (and above a floor of 1e-3 eps |G~|_F, which a rank-deficient G needs: its null-space entries are rounding noise).
// Record M | D | h | m | u_hat | k (p^2 + 5p doubles), M = R^-1 W column-major.  A chain that does not converge within
// EIG_MAX_SWEEPS or whose record is not finite gets D[0] = NaN: every draw of it is NaN with OMC_STATUS_NOT_PD.
//
// Draw (every sweep, one warp per chain): lane l owns coordinates 2l, 2l + 1 and the Philox block l of the chain, the
// normals the Cholesky kernels draw for the same coordinates (draw_z in dense_warp.cu).  beta = M u as p column loads of
// 16 bytes per lane (512 contiguous bytes per warp), EIG_COLS columns in flight.
#include "../../include/omc.h"
#include "omc_common.cuh"
#include "omc_internal.h"

#include <float.h>

namespace {

constexpr int EIG_PMAX = 64;
constexpr int PREP_THREADS = 256;
constexpr int EIG_MAX_SWEEPS = 40;
constexpr int DRAW_WARPS = 4;
constexpr int EIG_COLS = 8;

__device__ __forceinline__ double vat(const omc_vec_t& v, int chain, int i, double dflt) {
  return v.ptr ? v.ptr[(long long)chain * v.chain_stride + i] : dflt;
}

// sqrt of the prior precision's diagonal element i (kind 0: one value or NULL => 1)
__device__ __forceinline__ double prior_root(const omc_nn_eigen_prep_t& a, int chain, int i) {
  return sqrt(vat(a.prior_P, chain, a.prior_kind == OMC_MAT_DIAG ? i : 0, 1.0));
}

// Round r of the circle method over m (even) indices: pair k = (P, Q), P < Q; every pair appears once in m - 1 rounds
__device__ __forceinline__ void rr_pair(int m, int r, int k, int& P, int& Q) {
  int x, y;
  if (k == 0) {
    x = 0;
    y = 1 + r;
  } else {
    x = 1 + (r + k) % (m - 1);
    y = 1 + (r - k + m - 1) % (m - 1);
  }
  P = x < y ? x : y;
  Q = x < y ? y : x;
}

__global__ void __launch_bounds__(PREP_THREADS) nn_eigen_prep_kernel(omc_nn_eigen_prep_t a) {
  extern __shared__ __align__(16) double esm[];
  const int chain = blockIdx.x, tid = threadIdx.x, p = a.p;
  const int m = (p + 1) & ~1, h = m / 2, ld = m + 1;   // odd p: index p is a zero row / column, never rotated
  double* A = esm;                                     // G~ [m][ld]
  double* W = A + m * ld;                              // eigenvectors [m][ld]
  double* rt = W + m * ld;                             // sqrt(P0_ii) [m]
  double* rc = rt + m;                                 // rotation of pair k: c, s, t at 3k
  double* red = rc + 3 * (EIG_PMAX / 2);               // block-sum scratch [32]
  int* pq = reinterpret_cast<int*>(red + 32);          // P, Q of pair k at 2k
  int* flag = pq + EIG_PMAX;                           // [0] rotated in this sweep, [1] record bad

  const double* G = a.stats.ptr + (long long)chain * a.stats.chain_stride;
  if (tid < m) rt[tid] = tid < p ? prior_root(a, chain, tid) : 1.0;
  if (tid == 0) flag[1] = 0;
  __syncthreads();
  double fro = 0.0;
  for (int e = tid; e < m * m; e += PREP_THREADS) {
    const int i = e / m, j = e % m;
    double v = 0.0;
    if (i < p && j < p) v = (i >= j ? G[(long long)i * p + j] : G[(long long)j * p + i]) / (rt[i] * rt[j]);
    A[i * ld + j] = v;
    W[i * ld + j] = i == j ? 1.0 : 0.0;
    fro = fma(v, v, fro);
  }
  fro = sqrt(omc_block_sum(fro, red));
  const double floor_pq = 1e-3 * DBL_EPSILON * fro;

  bool converged = false;
  for (int sweep = 0; sweep < EIG_MAX_SWEEPS && !converged; ++sweep) {
    if (tid == 0) flag[0] = 0;
    __syncthreads();
    for (int r = 0; r < m - 1; ++r) {
      if (tid < h) {
        int P, Q;
        rr_pair(m, r, tid, P, Q);
        const double app = A[P * ld + P], aqq = A[Q * ld + Q], apq = A[P * ld + Q];
        double c = 1.0, s = 0.0, t = 0.0;
        if (fabs(apq) > DBL_EPSILON * sqrt(fabs(app * aqq)) && fabs(apq) > floor_pq) {
          const double th = (aqq - app) / (2.0 * apq);
          t = fabs(th) > 1e150 ? 0.5 / th : copysign(1.0, th) / (fabs(th) + sqrt(fma(th, th, 1.0)));
          c = 1.0 / sqrt(fma(t, t, 1.0));
          s = t * c;
          flag[0] = 1;
        }
        pq[2 * tid] = P;
        pq[2 * tid + 1] = Q;
        rc[3 * tid] = c;
        rc[3 * tid + 1] = s;
        rc[3 * tid + 2] = t;
      }
      __syncthreads();
      // A <- J'AJ: block (k, l), k <= l, rows P_k, Q_k and columns P_l, Q_l, mirrored into (l, k)
      for (int e = tid; e < h * h; e += PREP_THREADS) {
        const int k = e / h, l = e % h;
        if (k > l) continue;
        const int Pk = pq[2 * k], Qk = pq[2 * k + 1], Pl = pq[2 * l], Ql = pq[2 * l + 1];
        const double ck = rc[3 * k], sk = rc[3 * k + 1];
        if (k == l) {
          const double t = rc[3 * k + 2];
          if (t != 0.0) {
            const double apq = A[Pk * ld + Qk];
            A[Pk * ld + Pk] = fma(-t, apq, A[Pk * ld + Pk]);
            A[Qk * ld + Qk] = fma(t, apq, A[Qk * ld + Qk]);
            A[Pk * ld + Qk] = 0.0;
            A[Qk * ld + Pk] = 0.0;
          }
          continue;
        }
        const double cl = rc[3 * l], sl = rc[3 * l + 1];
        const double b00 = A[Pk * ld + Pl], b01 = A[Pk * ld + Ql], b10 = A[Qk * ld + Pl], b11 = A[Qk * ld + Ql];
        const double r00 = ck * b00 - sk * b10, r01 = ck * b01 - sk * b11;    // rows: J_k'
        const double r10 = sk * b00 + ck * b10, r11 = sk * b01 + ck * b11;
        const double n00 = cl * r00 - sl * r01, n01 = sl * r00 + cl * r01;    // columns: J_l
        const double n10 = cl * r10 - sl * r11, n11 = sl * r10 + cl * r11;
        A[Pk * ld + Pl] = n00; A[Pl * ld + Pk] = n00;
        A[Pk * ld + Ql] = n01; A[Ql * ld + Pk] = n01;
        A[Qk * ld + Pl] = n10; A[Pl * ld + Qk] = n10;
        A[Qk * ld + Ql] = n11; A[Ql * ld + Qk] = n11;
      }
      // W <- W J
      for (int e = tid; e < m * h; e += PREP_THREADS) {
        const int i = e / h, l = e % h;
        const double s = rc[3 * l + 1];
        if (s == 0.0) continue;
        const int Pl = pq[2 * l], Ql = pq[2 * l + 1];
        const double c = rc[3 * l], x = W[i * ld + Pl], y = W[i * ld + Ql];
        W[i * ld + Pl] = c * x - s * y;
        W[i * ld + Ql] = s * x + c * y;
      }
      __syncthreads();
    }
    converged = flag[0] == 0;
    __syncthreads();
  }

  // record: M (column-major, M[i][j] = W[i][j] / r_i) | D | h = W'R^-1 g | m = W'R mu0 | u_hat = W'R beta_hat | k = W'R^-1 c0
  const long long rl = (long long)p * p + 5ll * p;
  double* rec = a.eig + (long long)chain * rl;
  bool bad = !converged;
  for (int e = tid; e < p * p; e += PREP_THREADS) {
    const int j = e / p, i = e % p;
    const double v = W[i * ld + j] / rt[i];
    bad |= !isfinite(v);
    rec[e] = v;
  }
  const double* cen = a.center.ptr ? a.center.ptr + (long long)chain * a.center.chain_stride : nullptr;
  for (int e = tid; e < 5 * p; e += PREP_THREADS) {
    const int q = e / p, j = e % p;
    double v;
    if (q == 0) {
      v = A[j * ld + j];
    } else {
      v = 0.0;
      for (int i = 0; i < p; ++i) {
        double x;
        if (q == 1) x = G[(long long)p * p + i] / rt[i];
        else if (q == 2) x = vat(a.mu0, chain, i, 0.0) * rt[i];
        else if (q == 3) x = cen ? cen[i] * rt[i] : 0.0;
        else x = cen ? cen[p + i] / rt[i] : 0.0;
        v = fma(W[i * ld + j], x, v);
      }
    }
    bad |= !isfinite(v);
    rec[(long long)p * p + e] = v;
  }
  if (bad) flag[1] = 1;
  __syncthreads();
  if (tid == 0 && flag[1]) rec[(long long)p * p] = nan("");
}

// One warp per chain.  VEC: p even and the records 16-byte aligned (one double2 per lane and column).
template <bool VEC>
__global__ void __launch_bounds__(32 * DRAW_WARPS, 8) nn_eigen_draw_kernel(omc_nn_eigen_draw_t a) {
  const int chain = blockIdx.x * DRAW_WARPS + (threadIdx.x >> 5);
  if (chain >= a.n_chains) return;   // warp-uniform
  const int lane = threadIdx.x & 31, p = a.p;
  const int i0 = 2 * lane, i1 = i0 + 1;
  const bool own0 = i0 < p, own1 = i1 < p;
  const double* __restrict__ rec = a.eig + (long long)chain * ((long long)p * p + 5ll * p);
  const double* __restrict__ vD = rec + (long long)p * p;
  const double tau = vat(a.tau, chain, 0, 1.0), lam = vat(a.lambda, chain, 0, 1.0);

  double z0 = 0.0, z1 = 0.0;
  if (own0) {
    if (a.debug_z) {
      const double* dz = a.debug_z + (a.rng.sweep ? (long long)(*a.rng.sweep) : 0ll) * a.debug_sweep_stride + (long long)chain * p;
      z0 = dz[i0];
      if (own1) z1 = dz[i1];
    } else {
      OmcRng rg;
      rg.seed = a.rng.seed; rg.sweep = a.rng.sweep; rg.chain_offset = a.rng.chain_offset; rg.site = a.rng.site;
      omc_normal2(rg, chain, lane, z0, z1);
    }
  }
  // u = S^-1 (tau h + lam m) + S^-1/2 z; S must be positive and finite
  double u[2] = {0.0, 0.0};
  bool bad = false;
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int i = i0 + r;
    if (i < p) {
      const double S = fma(tau, vD[i], lam);
      if (!(S > 0.0) || !isfinite(S)) bad = true;
      u[r] = fma(tau, vD[p + i], lam * vD[2 * p + i]) / S + (r ? z1 : z0) / sqrt(S);
    }
  }
  double* beta = a.beta + (long long)chain * p;
  if (__any_sync(0xffffffffu, bad)) {
    if (lane == 0 && a.status) atomicOr(&a.status[chain], OMC_STATUS_NOT_PD);
    for (int c = lane; c < p; c += 32) beta[c] = nan("");
    return;
  }

  // beta = M u: column j of M is p contiguous doubles, lane l reads rows 2l, 2l + 1; u_j from lane j / 2
  double acc0 = 0.0, acc1 = 0.0;
  for (int j0 = 0; j0 < p; j0 += EIG_COLS) {
    double c0[EIG_COLS], c1[EIG_COLS];
#pragma unroll
    for (int jj = 0; jj < EIG_COLS; ++jj) {
      const int j = j0 + jj;
      c0[jj] = 0.0;
      c1[jj] = 0.0;
      if (j < p) {
        const double* col = rec + (long long)j * p;
        if (VEC) {
          if (own0) {
            const double2 v = __ldg(reinterpret_cast<const double2*>(col + i0));
            c0[jj] = v.x;
            c1[jj] = v.y;
          }
        } else {
          if (own0) c0[jj] = __ldg(col + i0);
          if (own1) c1[jj] = __ldg(col + i1);
        }
      }
    }
#pragma unroll
    for (int jj = 0; jj < EIG_COLS; ++jj) {
      const double uj = __shfl_sync(0xffffffffu, (jj & 1) ? u[1] : u[0], ((j0 + jj) >> 1) & 31);   // j0 is even
      acc0 = fma(c0[jj], uj, acc0);
      acc1 = fma(c1[jj], uj, acc1);
    }
  }
  if (own0) beta[i0] = acc0;
  if (own1) beta[i1] = acc1;

  if (a.center.ptr && a.rss_out) {
    // e'(D e - 2 k), e = u - u_hat
    double s = 0.0;
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int i = i0 + r;
      if (i < p) {
        const double e = u[r] - vD[3 * p + i];
        s = fma(e, fma(vD[i], e, -2.0 * vD[4 * p + i]), s);
      }
    }
    s = omc_warp_sum(s);
    if (lane == 0) a.rss_out[(long long)chain * a.rss_stride] = a.center.ptr[(long long)chain * a.center.chain_stride + 2 * p] + s;
  }
}

size_t prep_smem(int p) {
  const int m = (p + 1) & ~1;
  return (size_t)(2 * m * (m + 1) + m + 3 * (EIG_PMAX / 2) + 32) * sizeof(double) + (EIG_PMAX + 2) * sizeof(int);
}

}  // namespace

extern "C" int omc_nn_eigen_prep(const omc_nn_eigen_prep_t* args, void* stream) {
  OMC_REQUIRE(args && args->stats.ptr && args->eig, "omc_nn_eigen_prep: null argument");
  OMC_REQUIRE(args->p >= 1 && args->p <= EIG_PMAX, "omc_nn_eigen_prep: p=%d outside [1,%d]", args->p, EIG_PMAX);
  OMC_REQUIRE(args->n_chains >= 1, "omc_nn_eigen_prep: n_chains=%d", args->n_chains);
  OMC_REQUIRE(args->prior_kind == OMC_MAT_EYE || args->prior_kind == OMC_MAT_DIAG,
              "omc_nn_eigen_prep: prior_kind=%d (scaled identity or diagonal only)", args->prior_kind);
  OMC_REQUIRE(args->prior_kind == OMC_MAT_EYE || args->prior_P.ptr, "omc_nn_eigen_prep: prior_P missing");
  const size_t smem = prep_smem(args->p);
  OMC_CHECK_CUDA(cudaFuncSetAttribute(nn_eigen_prep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  nn_eigen_prep_kernel<<<args->n_chains, PREP_THREADS, smem, (cudaStream_t)stream>>>(*args);
  OMC_LAUNCH_CHECK();
  return 0;
}

extern "C" int omc_nn_eigen_draw(const omc_nn_eigen_draw_t* args, void* stream) {
  if (args) OMC_REQUIRE_SITE(args->rng, "omc_nn_eigen_draw");
  OMC_REQUIRE(args && args->eig && args->beta, "omc_nn_eigen_draw: null argument");
  OMC_REQUIRE(args->p >= 1 && args->p <= EIG_PMAX, "omc_nn_eigen_draw: p=%d outside [1,%d]", args->p, EIG_PMAX);
  OMC_REQUIRE(args->n_chains >= 1, "omc_nn_eigen_draw: n_chains=%d", args->n_chains);
  const unsigned grid = (unsigned)((args->n_chains + DRAW_WARPS - 1) / DRAW_WARPS);
  const bool vec = (args->p & 1) == 0 && (((unsigned long long)args->eig) & 15ull) == 0;
  if (vec) nn_eigen_draw_kernel<true><<<grid, 32 * DRAW_WARPS, 0, (cudaStream_t)stream>>>(*args);
  else nn_eigen_draw_kernel<false><<<grid, 32 * DRAW_WARPS, 0, (cudaStream_t)stream>>>(*args);
  OMC_LAUNCH_CHECK();
  return 0;
}
