// omc_nn_dense_draw for p <= 64 without probes: ONE WARP per chain.
//
//   Q = lambda*P0 + tau*G, L = chol(Q), x = L^-T (L^-1 b + z)          ref: sampler.py:154-207, gmrf.py:167-198, 29-61
//   (= mu + L^-T z with mu = L^-T L^-1 b, the reference's two solves folded into one backward substitution)
//
// Q is handled as 8 x 8 tiles in the accumulator layout of mma.sync.m8n8k4.f64: lane (g = lane / 4, kq = lane % 4)
// holds elements [g][2kq], [g][2kq+1] of a tile.  No CTA barrier: the CTA-wide kernels of the first round spent 40-55 %
// of a chain's life at barriers around their serial sections (profiles/r02_ncu_blocked64.txt).  Two forms:
//
// * Register kernel (nn_warp_draw_kernel, small p): the whole lower block triangle in registers (36 tiles = 72 doubles
//   per lane at p = 64), right-looking by block columns k (tools/gen/warp_chol_model.py is its lane-level numpy model):
//   the pivot stages of block column k (below), then the trailing update T(i, j) -= L(i, k) L(j, k)' as two
//   DMMA.8x8x4 per tile, the operand fragments being the panel tiles re-laid out inside their quads (4 shuffles per
//   tile).  At p = 64 it needs 254 registers per thread: 8 chains per SM.
// * Left-looking kernel (nn_left_draw_kernel, larger p; dense_draw.cu selects): only block column k in registers
//   (<= 16 doubles per lane, read from the record at the top of step k), the finished factor in the warp's slice of
//   shared memory.  Step k: C(i, k) = Q(i, k) - sum_{j<k} L(i, j) L(k, j)', i >= k, on the tensor pipe, summed from
//   zero with Q's tile added last (the record's latency hides behind the products); the products take a tile's k
//   index as 2kq + s in m8n8k4 step s, so both operand fragments are a lane's own accumulator element [g][2kq + s],
//   read as one 16-byte load per lane; the pivot stages of the diagonal tile alone, an identity tile riding along and
//   coming out as L_kk^-T; the panel L(i, k) = C(i, k) L_kk^-T as two DMMAs per tile straight from C's registers and
//   w[i] -= L(i, k) w[k] as a mat-vec; L(:, k), with L_kk^-1 in place of L_kk, back to shared memory; the rss epilogue
//   takes d from the backward solve's registers.  The backward solve is then one 8 x 8 mat-vec per block instead of 8 dependent substitution steps.  The pivot stages
//   no longer touch the off-diagonal tiles (224 of the 288 tile updates at p = 64, shuffle + 3 FMAs + select each).
//   At p = 64: 128 registers and 16,352 bytes of shared memory per warp, 14 chains per SM,
//   persistent warps, the next chain's record prefetched into L2 while the current one runs.  (A register copy of
//   block column k + 1 loaded one step ahead does not fit in the 128 registers: 4 of the 14 warps share one quarter
//   of the register file.)
//
// Pivot stages of block column k (register kernel): pivot from the diagonal tile by shuffle, 1/sqrt by MUFU.RSQ64H + two
// Newton steps, scale column, rank-1 update of the remaining columns of EVERY tile of the block column (independent work
// across the tiles hides the pivot chain); the right-hand side b (row layout, element 8i + g) rides along, so
// w = L^-1 b is there when the factorisation ends; 1/L_cc replaces L_cc on the diagonal.  The left-looking kernel runs
// the same stages on the diagonal tile only (factor_diag: L_kk and w[k] come out bit for bit the same).
// Backward solve L' x = w + z block by block from the bottom: partial sums of the off-diagonal products stay private
// per lane and are reduced over g (3 xor-shuffles) once per block; the 8 x 8 diagonal solves are quad-local
// substitutions (register kernel) or mat-vecs with L_jj^-1 (left-looking kernel).
// Epilogue: rss(beta) = rss0 - 2 d'c0 + d'G d from the centre record (omc.h), G read a second time (L2).
#include "../../include/omc.h"
#include "omc_common.cuh"
#include "omc_internal.h"

#include <utility>

namespace {

constexpr unsigned FULL = 0xffffffffu;
constexpr int WARPS_PER_CTA = 4;   // register kernel
constexpr int LL_WARPS = 14;       // left-looking kernel: one CTA of 14 warps per SM (448 threads x 128 registers)

__device__ __forceinline__ double wvec_at(const omc_vec_t& v, int chain, int i, double dflt) {
  return v.ptr ? v.ptr[(long long)chain * v.chain_stride + i] : dflt;
}
__device__ __forceinline__ double wrsqrt(double d) {
  double rd;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(rd) : "d"(d));
  const double hd = 0.5 * d;
  double e = fma(-hd, rd * rd, 0.5);
  rd = fma(rd, e, rd);
  e = fma(-hd, rd * rd, 0.5);
  return fma(rd, e, rd);   // 1/sqrt(d), relative error ~1e-16
}
__device__ __forceinline__ void wdmma(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}
__device__ __forceinline__ double shf(double v, int src) { return __shfl_sync(FULL, v, src); }
__device__ __forceinline__ double shx(double v, int m) { return __shfl_xor_sync(FULL, v, m); }

#define TI(i, j) ((i) * ((i) + 1) / 2 + (j))

template <int... K, class F>
__device__ __forceinline__ void static_for(std::integer_sequence<int, K...>, F f) {
  (f(std::integral_constant<int, K>{}), ...);
}

// Per-chain inputs of the draw
struct ChainIn {
  const double* rec;   // sufficient-statistics record: G (p x p) | g (p) | ...
  const double* P0;    // this chain's prior precision (null: identity)
  double tau, lam, diag_scale;
  bool dense;
};
__device__ __forceinline__ ChainIn chain_in(const omc_nn_dense_t& a, int chain) {
  ChainIn c;
  c.rec = a.stats.ptr + (long long)chain * a.stats.chain_stride;
  c.P0 = a.prior_P.ptr ? a.prior_P.ptr + (long long)chain * a.prior_P.chain_stride : nullptr;
  c.tau = wvec_at(a.tau, chain, 0, 1.0);
  c.lam = wvec_at(a.lambda, chain, 0, 1.0);
  c.diag_scale = a.mode == 1 ? 1.0 + a.ridge_rel : 1.0;
  c.dense = a.prior_kind == OMC_MAT_DENSE;
  return c;
}

// Elements [g][2kq], [g][2kq+1] of tile (i, j) of Q (sampler.py:180-186); rows / columns >= p are padded with the
// identity.  VEC: p even and a 16-byte aligned record, so col + 1 < p whenever col < p.
template <bool VEC>
__device__ __forceinline__ void q_pair(const omc_nn_dense_t& a, const ChainIn& ci, int p, int i, int j, int g, int kq,
                                       double& q0, double& q1) {
  const int row = 8 * i + g, col = 8 * j + 2 * kq;
  q0 = 0.0;
  q1 = 0.0;
  if (row < p) {
    if (VEC) {
      if (col < p) {
        const double2 v = *reinterpret_cast<const double2*>(ci.rec + (long long)row * p + col);
        q0 = ci.tau * v.x;
        q1 = ci.tau * v.y;
      }
    } else {
      if (col < p) q0 = ci.tau * ci.rec[(long long)row * p + col];
      if (col + 1 < p) q1 = ci.tau * ci.rec[(long long)row * p + col + 1];
    }
    if (ci.dense) {
      if (col < p) q0 = fma(ci.lam, ci.P0[(long long)row * p + col], q0);
      if (col + 1 < p) q1 = fma(ci.lam, ci.P0[(long long)row * p + col + 1], q1);
      if (i == j) {
        if (row == col) q0 *= ci.diag_scale;
        if (row == col + 1) q1 *= ci.diag_scale;
      }
    } else if (i == j) {
      const double pr = a.prior_kind == OMC_MAT_DIAG ? ci.P0[row] : (ci.P0 ? ci.P0[0] : 1.0);
      if (row == col) q0 = fma(ci.lam, pr, q0) * ci.diag_scale;
      if (row == col + 1) q1 = fma(ci.lam, pr, q1) * ci.diag_scale;
    }
  } else if (i == j) {
    if (row == col) q0 = 1.0;
    if (row == col + 1) q1 = 1.0;
  }
}

// b = (lam*P0) mu0 + tau*g in row layout: w[i] = element 8i + g (replicated over kq)
template <int PB>
__device__ __forceinline__ void rhs_rows(const omc_nn_dense_t& a, const ChainIn& ci, int p, int chain, int g,
                                         double (&w)[PB]) {
#pragma unroll
  for (int i = 0; i < PB; ++i) {
    const int row = 8 * i + g;
    double bc = 0.0;
    if (row < p) {
      double sacc;
      if (ci.dense) {
        sacc = 0.0;
        for (int j = 0; j < p; ++j) sacc += ci.lam * ci.P0[(long long)row * p + j] * wvec_at(a.mu0, chain, j, 0.0);
      } else {
        const double pr = a.prior_kind == OMC_MAT_DIAG ? ci.P0[row] : (ci.P0 ? ci.P0[0] : 1.0);
        sacc = ci.lam * pr * wvec_at(a.mu0, chain, row, 0.0);
      }
      bc = sacc + ci.tau * ci.rec[(long long)p * p + row];
    }
    w[i] = bc;
  }
}

// z: lane (g, kq) owns the pair of elements 8g + 2kq, +1 (Philox block = pair index, as in the other kernels)
template <int PB>
__device__ __forceinline__ void draw_z(const omc_nn_dense_t& a, int p, int chain, int g, int kq, double& z0, double& z1) {
  z0 = 0.0;
  z1 = 0.0;
  if (a.mode != 1 && g < PB) {
    const int e0 = 8 * g + 2 * kq;
    if (a.debug_z) {
      const double* dz = a.debug_z + (a.rng.sweep ? (long long)(*a.rng.sweep) : 0ll) * a.debug_sweep_stride + (long long)chain * p;
      if (e0 < p) z0 = dz[e0];
      if (e0 + 1 < p) z1 = dz[e0 + 1];
    } else if (e0 < p) {
      OmcRng rg;
      rg.seed = a.rng.seed; rg.sweep = a.rng.sweep; rg.chain_offset = a.rng.chain_offset; rg.site = a.rng.site;
      omc_normal2(rg, chain, 4 * g + kq, z0, z1);
      if (e0 + 1 >= p) z1 = 0.0;
    }
  }
}

// The 8 pivot stages of block column k on the panel tiles tile(i), i = k .. PB-1 (tile(i) -> double[2] in accumulator
// layout, tile(k) the diagonal one), with w riding along.  bad: a pivot was not positive (warp-uniform).
template <int PB, class Tile>
__device__ __forceinline__ void factor_panel(Tile tile, double (&w)[PB], int k, int g, int kq, bool& bad) {
#pragma unroll 1
  for (int jq = 0; jq < 4; ++jq) {
    const bool own = kq == jq;
#pragma unroll
    for (int reg = 0; reg < 2; ++reg) {
      const int jj = 2 * jq + reg;
      double* D = tile(k);
      const double piv = shf(D[reg], 4 * jj + jq);
      if (!(piv > 0.0)) bad = true;
      const double rd = wrsqrt(piv);
#pragma unroll
      for (int i = k; i < PB; ++i) tile(i)[reg] = own ? tile(i)[reg] * rd : tile(i)[reg];
      const double wc = shf(w[k], 4 * jj) * rd;
      if (g == jj) w[k] = wc;
      double lc0 = shf(D[reg], 8 * kq + jq);        // L[2kq][jj]
      double lc1 = shf(D[reg], 8 * kq + 4 + jq);    // L[2kq+1][jj]
      if (!(2 * kq > jj)) lc0 = 0.0;
      if (!(2 * kq + 1 > jj)) lc1 = 0.0;
#pragma unroll
      for (int i = k; i < PB; ++i) {
        double* T = tile(i);
        const double lg = shf(T[reg], 4 * g + jq);  // L[8i + g][8k + jj]
        T[0] = fma(-lg, lc0, T[0]);
        T[1] = fma(-lg, lc1, T[1]);
        if (i == k) {
          if (g > jj) w[k] = fma(-lg, wc, w[k]);
        } else {
          w[i] = fma(-lg, wc, w[i]);
        }
      }
      if (own && g == jj) D[reg] = rd;              // 1 / L_cc on the diagonal from here on
    }
  }
}

// The pivot stages of the diagonal tile D = C(k, k) alone, with w[k] riding along: D and w[k] come out exactly as from
// factor_panel.  E enters as the identity and sees the same column operations, so it leaves as L_kk^-T (upper
// triangular, exact zeros below the diagonal) in accumulator layout.  D's diagonal keeps L_cc: nothing reads D again.
__device__ __forceinline__ void factor_diag(double (&D)[2], double (&E)[2], double& wk, int g, int kq, bool& bad) {
#pragma unroll 1
  for (int jq = 0; jq < 4; ++jq) {
    const bool own = kq == jq;
#pragma unroll
    for (int reg = 0; reg < 2; ++reg) {
      const int jj = 2 * jq + reg;
      const double piv = shf(D[reg], 4 * jj + jq);
      if (!(piv > 0.0)) bad = true;
      const double rd = wrsqrt(piv);
      D[reg] = own ? D[reg] * rd : D[reg];
      E[reg] = own ? E[reg] * rd : E[reg];
      const double wc = shf(wk, 4 * jj) * rd;
      if (g == jj) wk = wc;
      double lc0 = shf(D[reg], 8 * kq + jq);        // L[2kq][jj]
      double lc1 = shf(D[reg], 8 * kq + 4 + jq);    // L[2kq+1][jj]
      if (!(2 * kq > jj)) lc0 = 0.0;
      if (!(2 * kq + 1 > jj)) lc1 = 0.0;
      const double lg = shf(D[reg], 4 * g + jq);    // L[g][jj]
      const double le = shf(E[reg], 4 * g + jq);    // E[g][jj]
      D[0] = fma(-lg, lc0, D[0]);
      D[1] = fma(-lg, lc1, D[1]);
      if (g > jj) wk = fma(-lg, wc, wk);
      E[0] = fma(-le, lc0, E[0]);
      E[1] = fma(-le, lc1, E[1]);
    }
  }
}

// r = w + z in column layout; racc = per-lane partial sums of the backward solve (the g == 0 lanes start from r)
template <int PB>
__device__ __forceinline__ void solve_rhs(double (&racc)[PB][2], const double (&w)[PB], double z0, double z1, int g,
                                          int kq) {
#pragma unroll
  for (int tc = 0; tc < PB; ++tc)
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const double wcol = shf(w[tc], 4 * (2 * kq + r));
      const double zcol = shf(r ? z1 : z0, 4 * tc + kq);
      racc[tc][r] = (g == 0) ? wcol + zcol : 0.0;
    }
}

// Backward solve L' x = w + z, x -> beta.  ldiag(j, c, l0, l1): L_jj[c][2kq], L_jj[c][2kq+1] (1 / L_cc on the
// diagonal; only the lower triangle is used); loff(j, tc, r): L(j, tc)[g][2kq + r], tc < j.
template <int PB, class Diag, class Off>
__device__ __forceinline__ void back_solve(double* beta, int p, const double (&w)[PB], double z0, double z1, int g, int kq,
                                           Diag ldiag, Off loff) {
  double racc[PB][2];
  solve_rhs<PB>(racc, w, z0, z1, g, kq);
#pragma unroll
  for (int j = PB - 1; j >= 0; --j) {
    double v0 = racc[j][0], v1 = racc[j][1];
    v0 += shx(v0, 4); v1 += shx(v1, 4);
    v0 += shx(v0, 8); v1 += shx(v1, 8);
    v0 += shx(v0, 16); v1 += shx(v1, 16);
#pragma unroll 1
    for (int cq = 3; cq >= 0; --cq) {
#pragma unroll
      for (int reg = 1; reg >= 0; --reg) {
        const int c = 2 * cq + reg;
        double l0, l1;
        ldiag(j, c, l0, l1);
        const double mine = reg ? v1 * l1 : v0 * l0;
        const double xc = shf(mine, 4 * g + cq);
        if (kq == cq) { if (reg) v1 = xc; else v0 = xc; }
        if (2 * kq < c) v0 = fma(-l0, xc, v0);
        if (2 * kq + 1 < c) v1 = fma(-l1, xc, v1);
      }
    }
    if (g == 0) {
      const int e0 = 8 * j + 2 * kq;
      if (e0 < p) beta[e0] = v0;
      if (e0 + 1 < p) beta[e0 + 1] = v1;
    }
    if (j > 0) {
      const double a0 = shf(v0, 4 * g + (g >> 1)), a1 = shf(v1, 4 * g + (g >> 1));
      const double xg = (g & 1) ? a1 : a0;                      // x[8j + g]
#pragma unroll
      for (int tc = 0; tc < j; ++tc) {
        racc[tc][0] = fma(-loff(j, tc, 0), xg, racc[tc][0]);
        racc[tc][1] = fma(-loff(j, tc, 1), xg, racc[tc][1]);
      }
    }
  }
}

// Backward solve L' x = w + z with the inverted diagonal blocks, x -> beta: x_j = L_jj^-T v_j is one 8 x 8 mat-vec
// (lane-local) and a quad reduction, which leaves x_j in row layout (x[8j + g]), the form the off-diagonal updates
// take.  linv(j, l0, l1): L_jj^-1[2kq][g], L_jj^-1[2kq+1][g] (0 above the diagonal); loff(j, tc): L(j, tc)[g][2kq],
// L(j, tc)[g][2kq + 1] as one double2, tc < j.  xr[j] = x[8j + g] stays behind for the rss epilogue.
template <int PB, class Inv, class Off>
__device__ __forceinline__ void back_solve_inv(double* beta, int p, const double (&w)[PB], double z0, double z1, int g,
                                               int kq, Inv linv, Off loff, double (&xr)[PB]) {
  double racc[PB][2];
  solve_rhs<PB>(racc, w, z0, z1, g, kq);
#pragma unroll
  for (int j = PB - 1; j >= 0; --j) {
    double v0 = racc[j][0], v1 = racc[j][1];
    v0 += shx(v0, 4); v1 += shx(v1, 4);
    v0 += shx(v0, 8); v1 += shx(v1, 8);
    v0 += shx(v0, 16); v1 += shx(v1, 16);
    double l0, l1;
    linv(j, l0, l1);
    double xg = fma(l0, v0, l1 * v1);
    xg += shx(xg, 1);
    xg += shx(xg, 2);                                           // x[8j + g], the same bits in all four lanes
    if (kq == 0 && 8 * j + g < p) beta[8 * j + g] = xg;
    xr[j] = xg;
#pragma unroll
    for (int tc = 0; tc < j; ++tc) {
      const double2 l = loff(j, tc);
      racc[tc][0] = fma(-l.x, xg, racc[tc][0]);
      racc[tc][1] = fma(-l.y, xg, racc[tc][1]);
    }
  }
}

// Not positive definite: beta = 0 in solve-only mode (the centre may be any point: fall back to the origin), else NaN
// and the status flag
__device__ __forceinline__ void not_pd(const omc_nn_dense_t& a, int chain, double* beta, int lane) {
  if (a.mode == 1) {
    for (int c = lane; c < a.p; c += 32) beta[c] = 0.0;
    return;
  }
  if (lane == 0 && a.status) atomicOr(&a.status[chain], OMC_STATUS_NOT_PD);
  for (int c = lane; c < a.p; c += 32) beta[c] = nan("");
}

// rss(beta) = rss0 - 2 d'c0 + d'G d  (omc.h), d = beta - beta_hat from the centre record cen, G from the record again
// (not as |L'd|^2 - lam d'P0 d, which would carry the factorisation's backward error, ~cond(Q)).  dcol[j][r] =
// d[8j + 2kq + r], drow[j] = d[8j + g], 0 past p.
template <int PB, bool VEC>
__device__ __forceinline__ void rss_sum(const omc_nn_dense_t& a, int p, int chain, const double* __restrict__ rec,
                                        const double* cen, const double (&dcol)[PB][2], const double (&drow)[PB],
                                        int lane) {
  const int g = lane >> 2, kq = lane & 3;
  double acc = 0.0;
#pragma unroll
  for (int j = 0; j < PB; ++j) {
    const int e0 = 8 * j + 2 * kq;
    if (g == 0) {
      if (e0 < p) acc = fma(-2.0 * cen[p + e0], dcol[j][0], acc);
      if (e0 + 1 < p) acc = fma(-2.0 * cen[p + e0 + 1], dcol[j][1], acc);
    }
  }
#pragma unroll
  for (int i = 0; i < PB; ++i)
#pragma unroll
    for (int j = 0; j <= i; ++j) {
      const int row = 8 * i + g, col = 8 * j + 2 * kq;
      double g0 = 0.0, g1 = 0.0;
      if (row < p) {
        if (VEC) {
          if (col < p) {
            const double2 v = *reinterpret_cast<const double2*>(rec + (long long)row * p + col);
            g0 = v.x;
            g1 = v.y;
          }
        } else {
          if (col < p) g0 = rec[(long long)row * p + col];
          if (col + 1 < p) g1 = rec[(long long)row * p + col + 1];
        }
      }
      const double t = fma(g0, dcol[j][0], g1 * dcol[j][1]) * drow[i];
      acc += (i == j) ? t : 2.0 * t;
    }
  acc = omc_warp_sum(acc);
  if (lane == 0) a.rss_out[(long long)chain * a.stats.chain_stride] = cen[2 * p] + acc;
}

// rss epilogue of the register kernel: beta is read back through L2
template <int PB, bool VEC>
__device__ __forceinline__ void rss_epilogue(const omc_nn_dense_t& a, int p, int chain, const double* __restrict__ rec,
                                             const double* beta, int lane) {
  const int g = lane >> 2, kq = lane & 3;
  __syncwarp();
  const double* cen = a.center.ptr + (long long)chain * a.center.chain_stride;
  double dcol[PB][2], drow[PB];
#pragma unroll
  for (int j = 0; j < PB; ++j) {
    const int e0 = 8 * j + 2 * kq, er = 8 * j + g;
    dcol[j][0] = e0 < p ? __ldcg(beta + e0) - cen[e0] : 0.0;
    dcol[j][1] = e0 + 1 < p ? __ldcg(beta + e0 + 1) - cen[e0 + 1] : 0.0;
    drow[j] = er < p ? __ldcg(beta + er) - cen[er] : 0.0;
  }
  rss_sum<PB, VEC>(a, p, chain, rec, cen, dcol, drow, lane);
}

// ---------------------------------------------------------------------------------------------------------------------
// Register kernel: one chain, one warp, the lower block triangle of Q in registers.
template <int PB, bool VEC>
__device__ __forceinline__ void warp_chain(const omc_nn_dense_t& a, int chain) {
  const int lane = threadIdx.x & 31;
  const int g = lane >> 2, kq = lane & 3, p = a.p;
  const ChainIn ci = chain_in(a, chain);

  double T[PB * (PB + 1) / 2][2];
#pragma unroll
  for (int i = 0; i < PB; ++i)
#pragma unroll
    for (int j = 0; j <= i; ++j) q_pair<VEC>(a, ci, p, i, j, g, kq, T[TI(i, j)][0], T[TI(i, j)][1]);
  double w[PB];
  rhs_rows<PB>(a, ci, p, chain, g, w);
  double z0, z1;
  draw_z<PB>(a, p, chain, g, kq, z0, z1);

  // ---- factorisation by block columns, right-looking
  bool bad = false;
#pragma unroll
  for (int k = 0; k < PB; ++k) {
    factor_panel<PB>([&](int i) -> double* { return T[TI(i, k)]; }, w, k, g, kq, bad);
    if (k + 1 < PB) {
      // panel tiles as operand fragments: f_s = element [g][4s + kq] (quad-local re-layout)
      double R[PB][2];
#pragma unroll
      for (int i = k + 1; i < PB; ++i)
#pragma unroll
        for (int s = 0; s < 2; ++s) {
          const int src = 4 * g + 2 * s + (kq >> 1);
          const double v0 = shf(T[TI(i, k)][0], src), v1 = shf(T[TI(i, k)][1], src);
          R[i][s] = (kq & 1) ? v1 : v0;
        }
#pragma unroll
      for (int j = k + 1; j < PB; ++j)
#pragma unroll
        for (int i = j; i < PB; ++i) {
          wdmma(T[TI(i, j)][0], T[TI(i, j)][1], -R[i][0], R[j][0]);
          wdmma(T[TI(i, j)][0], T[TI(i, j)][1], -R[i][1], R[j][1]);
        }
    }
  }
  double* beta = a.beta + (long long)chain * p;
  if (bad) return not_pd(a, chain, beta, lane);
  back_solve<PB>(
      beta, p, w, z0, z1, g, kq,
      [&](int j, int c, double& l0, double& l1) {
        l0 = shf(T[TI(j, j)][0], 4 * c + kq);
        l1 = shf(T[TI(j, j)][1], 4 * c + kq);
      },
      [&](int j, int tc, int r) { return T[TI(j, tc)][r]; });
  if (a.center.ptr && a.rss_out) rss_epilogue<PB, VEC>(a, p, chain, ci.rec, beta, lane);
}

// resident CTAs (of 4 warps) per SM the register allocation aims at: 72 doubles of tiles per lane at PB = 8
template <int PB>
constexpr int ctas_per_sm() { return PB <= 2 ? 5 : (PB <= 4 ? 3 : 2); }

template <int PB, bool VEC>
__global__ void __launch_bounds__(32 * WARPS_PER_CTA, ctas_per_sm<PB>()) nn_warp_draw_kernel(omc_nn_dense_t a) {
  const int chain = blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5);
  if (chain < a.n_chains) warp_chain<PB, VEC>(a, chain);   // warp-uniform
}

// ---------------------------------------------------------------------------------------------------------------------
// Left-looking kernel.  Shared-memory slice of one warp: the PB(PB-1)/2 off-diagonal tiles of L full, then the PB-1
// first diagonal blocks' INVERSES L_kk^-1 as packed lower triangles (36 doubles, element [r][c] at r(r+1)/2 + c; the
// backward solve is their only reader); the last one stays in registers, as L_77^-T in accumulator layout.
// An off-diagonal tile is stored in accumulator layout, lane l's two elements ([g][2kq], [g][2kq + 1]) at 2l, 2l + 1:
// one 16-byte store or load per lane, 512 contiguous bytes per warp.  The products take the tile's k index in the
// order k = 2kq + s in m8n8k4 step s, so that a lane's operand fragment of step s is its own element [g][2kq + s].
template <int PB>
struct LeftSmem {
  static constexpr int DIAG_OFF = 64 * (PB * (PB - 1) / 2);
  static constexpr int DOUBLES = DIAG_OFF + 36 * (PB - 1);                // 2044 at PB = 8
  __host__ __device__ static constexpr int off(int i, int j) { return 64 * (i * (i - 1) / 2 + j); }   // tile (i, j), i > j
};

// FULL: p = 8 PB and a 16-byte aligned record (16-byte loads, every bound known at compile time); else any p of the
// block count, element by element
template <int PB, bool FULL>
__device__ __forceinline__ void left_chain(const omc_nn_dense_t& a, int chain, int next_chain, double* sm) {
  using S = LeftSmem<PB>;
  constexpr bool VEC = FULL;
  const int lane = threadIdx.x & 31;
  const int g = lane >> 2, kq = lane & 3, p = FULL ? 8 * PB : a.p;
  const ChainIn ci = chain_in(a, chain);

  // the next chain's record (and centre record) on its way into L2 while this one runs; every byte of both is read
  if (VEC && next_chain >= 0) {
    const char* nrec = reinterpret_cast<const char*>(a.stats.ptr + (long long)next_chain * a.stats.chain_stride);
    const unsigned bytes = 8u * (unsigned)(p * p + p);                   // p (p + 1) is even: a multiple of 16
    const unsigned chunk = ((bytes + 32u * 16u - 1u) / (32u * 16u)) * 16u;
    const unsigned o = chunk * (unsigned)lane;
    if (o < bytes) {
      const unsigned n = bytes - o < chunk ? bytes - o : chunk;
      asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;\n" ::"l"(nrec + o), "r"(n) : "memory");
    }
    const double* ncen = a.center.ptr + (long long)next_chain * a.center.chain_stride;
    if (lane == 0 && a.center.ptr && a.rss_out && (((unsigned long long)ncen) & 15ull) == 0)
      asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;\n" ::"l"(ncen),
                   "r"(16u * (unsigned)(p + 1))
                   : "memory");
  }

  double C[PB][2];   // block column k: C[i] = tile (i, k), i >= k
  double E[2];       // L_kk^-T of the current step (of the last one, for the backward solve)
  double w[PB];
  rhs_rows<PB>(a, ci, p, chain, g, w);
  double z0, z1;     // drawn in the last step, in the issue gaps of its pivot stages (earlier they would spill)
  __syncwarp();      // the previous chain's reads of the slice are done

  bool bad = false;
  // the steps are unrolled by hand: every register array must be indexed by constants
  static_for(std::make_integer_sequence<int, PB>{}, [&](auto kc) {
    constexpr int k = decltype(kc)::value;
    // block column k of Q from the record (in L2 by now), added once the products are summed: its latency overlaps
    // the whole j loop instead of holding up the first DMMA
    double q[PB][2];
#pragma unroll
    for (int i = k; i < PB; ++i) q_pair<VEC>(a, ci, p, i, k, g, kq, q[i][0], q[i][1]);
    // C(i, k) = Q(i, k) - sum_j L(i, j) L(k, j)', j < k: in step s, A = element [g][2kq + s] of L(i, j), B the same
    // element of L(k, j)
#pragma unroll
    for (int i = k; i < PB; ++i) C[i][0] = C[i][1] = 0.0;
#pragma unroll
    for (int j = 0; j < k; ++j) {
      const double2 bk = *reinterpret_cast<const double2*>(sm + S::off(k, j) + 2 * lane);
      wdmma(C[k][0], C[k][1], -bk.x, bk.x);
      wdmma(C[k][0], C[k][1], -bk.y, bk.y);
#pragma unroll
      for (int i = k + 1; i < PB; ++i) {
        const double2 ai = *reinterpret_cast<const double2*>(sm + S::off(i, j) + 2 * lane);
        wdmma(C[i][0], C[i][1], -ai.x, bk.x);
        wdmma(C[i][0], C[i][1], -ai.y, bk.y);
      }
    }
#pragma unroll
    for (int i = k; i < PB; ++i) {
      C[i][0] += q[i][0];
      C[i][1] += q[i][1];
    }
    if (k == PB - 1) draw_z<PB>(a, p, chain, g, kq, z0, z1);
    E[0] = g == 2 * kq ? 1.0 : 0.0;
    E[1] = g == 2 * kq + 1 ? 1.0 : 0.0;
    factor_diag(C[k], E, w[k], g, kq, bad);
    if (k + 1 < PB) {
      // B fragments of E = L_kk^-T: step s needs E[2kq + s][g], held by lane (2kq + s, g >> 1), register g & 1
      double bf[2];
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        const int src = 4 * (2 * kq + s) + (g >> 1);
        const double e0 = shf(E[0], src), e1 = shf(E[1], src);
        bf[s] = (g & 1) ? e1 : e0;
      }
      const double wk0 = shf(w[k], 8 * kq), wk1 = shf(w[k], 8 * kq + 4);   // w[k] at 2kq, 2kq + 1
#pragma unroll
      for (int i = k + 1; i < PB; ++i) {
        // L(i, k) = C(i, k) L_kk^-T: A of step s = the lane's own element [g][2kq + s] of C(i, k)
        double l0 = 0.0, l1 = 0.0;
        wdmma(l0, l1, C[i][0], bf[0]);
        wdmma(l0, l1, C[i][1], bf[1]);
        *reinterpret_cast<double2*>(sm + S::off(i, k) + 2 * lane) = make_double2(l0, l1);
        // w[i] -= L(i, k) w[k]
        double t = fma(l0, wk0, l1 * wk1);
        t += shx(t, 1);
        t += shx(t, 2);
        w[i] -= t;
      }
      // L_kk^-1 as a packed lower triangle: element [r][c] = E[c][r], r = 2kq + e, c = g
      double* dt = sm + S::DIAG_OFF + 36 * k + g;
      if (2 * kq >= g) dt[kq * (2 * kq + 1)] = E[0];
      if (2 * kq + 1 >= g) dt[(2 * kq + 1) * (kq + 1)] = E[1];
      __syncwarp();
    }
  });
  double* beta = a.beta + (long long)chain * p;
  if (bad) return not_pd(a, chain, beta, lane);
  // the centre record's beta_hat in row layout, on its way while the backward solve runs
  const bool rss = a.center.ptr && a.rss_out;
  const double* cen = a.center.ptr + (long long)chain * a.center.chain_stride;
  double crow[PB];
#pragma unroll
  for (int j = 0; j < PB; ++j) crow[j] = rss && 8 * j + g < p ? cen[8 * j + g] : 0.0;
  double xr[PB];
  back_solve_inv<PB>(
      beta, p, w, z0, z1, g, kq,
      [&](int j, double& l0, double& l1) {
        if (j == PB - 1) {                            // E of the last step is L_77^-T: E[g][2kq + e] = L_77^-1[2kq + e][g]
          l0 = E[0];
          l1 = E[1];
        } else {
          const double* dt = sm + S::DIAG_OFF + 36 * j + g;
          l0 = 2 * kq >= g ? dt[kq * (2 * kq + 1)] : 0.0;
          l1 = 2 * kq + 1 >= g ? dt[(2 * kq + 1) * (kq + 1)] : 0.0;
        }
      },
      [&](int j, int tc) { return *reinterpret_cast<const double2*>(sm + S::off(j, tc) + 2 * lane); }, xr);
  if (rss) {
    // d from the solve's own registers: drow[j] = x[8j + g] - beta_hat[8j + g], the column layout by shuffle (the
    // same doubles, with no store -> load round trip through L2)
    double dcol[PB][2], drow[PB];
#pragma unroll
    for (int j = 0; j < PB; ++j) drow[j] = 8 * j + g < p ? xr[j] - crow[j] : 0.0;
#pragma unroll
    for (int j = 0; j < PB; ++j) {
      dcol[j][0] = shf(drow[j], 8 * kq);
      dcol[j][1] = shf(drow[j], 8 * kq + 4);
    }
    rss_sum<PB, VEC>(a, p, chain, ci.rec, cen, dcol, drow, lane);
  }
}

template <int PB, bool FULL>
__global__ void __launch_bounds__(32 * LL_WARPS, 1) nn_left_draw_kernel(omc_nn_dense_t a) {
  extern __shared__ __align__(16) double dsm[];
  const int wid = threadIdx.x >> 5;
  const int n_warps = gridDim.x * LL_WARPS;
  double* sm = dsm + wid * LeftSmem<PB>::DOUBLES;
  for (int chain = blockIdx.x * LL_WARPS + wid; chain < a.n_chains; chain += n_warps) {   // warp-uniform
    const int nxt = chain + n_warps;
    left_chain<PB, FULL>(a, chain, nxt < a.n_chains ? nxt : -1, sm);
  }
}

bool vec_ok(const omc_nn_dense_t& a) {
  return (a.p & 1) == 0 && (((unsigned long long)a.stats.ptr) & 15ull) == 0 && (a.stats.chain_stride & 1) == 0;
}

template <int PB>
int launch_warp_pb(const omc_nn_dense_t& a, cudaStream_t st) {
  const unsigned grid = (unsigned)((a.n_chains + WARPS_PER_CTA - 1) / WARPS_PER_CTA);
  if (vec_ok(a)) nn_warp_draw_kernel<PB, true><<<grid, 32 * WARPS_PER_CTA, 0, st>>>(a);
  else nn_warp_draw_kernel<PB, false><<<grid, 32 * WARPS_PER_CTA, 0, st>>>(a);
  OMC_LAUNCH_CHECK();
  return 0;
}

template <int PB, bool FULL>
int launch_left(const omc_nn_dense_t& a, unsigned grid, cudaStream_t st) {
  const int smem = LL_WARPS * LeftSmem<PB>::DOUBLES * (int)sizeof(double);
  OMC_CHECK_CUDA(cudaFuncSetAttribute(nn_left_draw_kernel<PB, FULL>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  nn_left_draw_kernel<PB, FULL><<<grid, 32 * LL_WARPS, smem, st>>>(a);
  OMC_LAUNCH_CHECK();
  return 0;
}

template <int PB>
int launch_left_pb(const omc_nn_dense_t& a, cudaStream_t st) {
  // persistent warps: one CTA of 14 warps per SM
  const int ctas_needed = (a.n_chains + LL_WARPS - 1) / LL_WARPS;
  const int sms = omc_sm_count();
  const unsigned grid = (unsigned)(ctas_needed < sms ? ctas_needed : sms);
  return vec_ok(a) && a.p == 8 * PB ? launch_left<PB, true>(a, grid, st) : launch_left<PB, false>(a, grid, st);
}

}  // namespace

int omc_launch_warp_draw(const omc_nn_dense_t& a, cudaStream_t st) {
  switch ((a.p + 7) / 8) {
    case 1: return launch_warp_pb<1>(a, st);
    case 2: return launch_warp_pb<2>(a, st);
    case 3: return launch_warp_pb<3>(a, st);
    case 4: return launch_warp_pb<4>(a, st);
    case 5: return launch_warp_pb<5>(a, st);
    case 6: return launch_warp_pb<6>(a, st);
    case 7: return launch_warp_pb<7>(a, st);
    default: return launch_warp_pb<8>(a, st);
  }
}

int omc_launch_left_draw(const omc_nn_dense_t& a, cudaStream_t st) {   // 40 < p <= 64 (dense_draw.cu: LEFT_MIN_P)
  switch ((a.p + 7) / 8) {
    case 6: return launch_left_pb<6>(a, st);
    case 7: return launch_left_pb<7>(a, st);
    default: return launch_left_pb<8>(a, st);
  }
}
