// Blocked right-looking Cholesky of an augmented matrix [A ; b'] with an FP64 tensor-core (DMMA) trailing update and the
// backward solves that go with it, one CTA per matrix.  Shared by the dense conjugate draw / stand-alone factorisation
// (dense_blocked.cu, whose header comment describes the storage and the three steps per panel) and the ManifoldMALA step
// above 64 parameters (mh.cu).  Included inside each translation unit's anonymous namespace.
#pragma once

constexpr int NB = 16;           // panel width
constexpr int PLD = NB + 4;      // leading dimension of the panel buffer (== 4 mod 16: conflict-free fragment reads)
constexpr int SDLD = NB + 1;

__device__ __forceinline__ double rsqrt_newton(double d) {
  double rd;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(rd) : "d"(d));
  const double hd = 0.5 * d;
  double e = fma(-hd, rd * rd, 0.5);
  rd = fma(rd, e, rd);
  e = fma(-hd, rd * rd, 0.5);
  return fma(rd, e, rd);   // 1/sqrt(d), relative error ~1e-16
}
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

struct Workspace {
  double* A;      // (rows_pad x LD) augmented matrix, lower triangle
  double* Pn;     // (rows_pad x PLD) current panel, rows below the diagonal block
  double* sD;     // NB x SDLD factored diagonal block
  double* sinv;   // 1 / L_jj
  int LD, rows_pad;
};

// Factorises the leading p x p lower triangle of A in place and forward-solves the n_extra rows below it
// (rows p .. p+n_extra-1 become  row * L^-T, i.e. L^-1 b for a right-hand side stored as a row).
// Returns false (uniformly over the CTA) if a pivot was not positive; *s_bad must be zero on entry.
template <int NT>
__device__ bool blocked_cholesky(const Workspace& W, int p, int n_extra, int* s_bad) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NW = NT / 32;
  const int LD = W.LD;
  double* A = W.A;
  const int n_rows = p + n_extra;
  for (int k0 = 0; k0 < p; k0 += NB) {
    const int nbk = min(NB, p - k0), k1 = k0 + nbk;
    // ---- 1. diagonal block: warp 0, lane = row of the block
    if (warp == 0) {
      double d[NB];
      const int row = k0 + lane;
#pragma unroll
      for (int m = 0; m < NB; ++m) d[m] = (lane < nbk && m <= lane) ? A[(long long)row * LD + k0 + m] : 0.0;
      bool bad = false;
#pragma unroll
      for (int j = 0; j < NB; ++j) {
        if (j < nbk) {                                        // uniform
          const double piv = __shfl_sync(0xffffffffu, d[j], j);
          if (!(piv > 0.0)) bad = true;
          const double rd = rsqrt_newton(piv);
          const double lj = (lane == j) ? piv * rd : d[j] * rd;   // L[row][k0 + j]
          d[j] = lj;
          if (lane == j) W.sinv[k0 + j] = rd;
#pragma unroll
          for (int m = j + 1; m < NB; ++m) {
            const double v = __shfl_sync(0xffffffffu, lj, m);     // L[k0 + m][k0 + j]
            d[m] = fma(-lj, v, d[m]);
          }
        }
      }
      if (bad && lane == 0) *s_bad = 1;
      if (lane < nbk) {
#pragma unroll
        for (int m = 0; m < NB; ++m)
          if (m <= lane) {
            A[(long long)row * LD + k0 + m] = d[m];
            W.sD[lane * SDLD + m] = d[m];
          }
      }
    }
    __syncthreads();
    if (*s_bad) return false;
    // ---- 2. rows below the block: x L11' = a  (one thread per row, forward substitution over the 16 columns)
    for (int r = k1 + tid; r < n_rows; r += NT) {
      double x[NB];
      double* arow = A + (long long)r * LD + k0;
#pragma unroll
      for (int j = 0; j < NB; ++j) x[j] = (j < nbk) ? arow[j] : 0.0;
#pragma unroll
      for (int j = 0; j < NB; ++j) {
        if (j < nbk) {
          double s = x[j];
#pragma unroll
          for (int m = 0; m < j; ++m) s = fma(-x[m], W.sD[j * SDLD + m], s);
          x[j] = s * W.sinv[k0 + j];
        }
      }
#pragma unroll
      for (int j = 0; j < NB; ++j) {
        if (j < nbk) arow[j] = x[j];
        W.Pn[r * PLD + j] = x[j];
      }
    }
    __syncthreads();
    // ---- 3. trailing update on the FP64 tensor pipe: C(ti, tj) -= P(ti) P(tj)' over the lower-triangle 8 x 8 tiles
    if (k1 < p) {
      const int T0 = k1 >> 3;                               // k1 is a multiple of 16 here
      const int Tr = (W.rows_pad >> 3) - T0, Tc = ((p + 7) >> 3) - T0;
      const int g = lane >> 2, kq = lane & 3;
      // this warp's tiles (round-robin over the row-major enumeration of the lower triangle), four at a time: the C
      // loads of a batch go out together and its 16 DMMAs interleave (a store -> load pair per tile would serialise
      // them: the compiler cannot prove that Pn and A do not alias)
      constexpr int TB = 4;
      int ti = 0, tj = 0, idx = 0;
      const long long total = (long long)Tc * (Tc + 1) / 2 + (long long)(Tr - Tc) * Tc;
      auto advance = [&]() {
        ++idx;
        if (++tj > min(ti, Tc - 1)) { tj = 0; ++ti; }
      };
      while (idx < total && (idx & (NW - 1)) != warp) advance();
      while (idx < total) {
        double2* pc[TB];
        const double* pa[TB];
        const double* pb[TB];
        double2 c[TB];
        int nb = 0;
#pragma unroll
        for (int q = 0; q < TB; ++q) {
          if (idx < total) {
            pa[q] = W.Pn + (8 * (T0 + ti) + g) * PLD + kq;
            pb[q] = W.Pn + (8 * (T0 + tj) + g) * PLD + kq;
            pc[q] = reinterpret_cast<double2*>(A + (long long)(8 * (T0 + ti) + g) * LD + 8 * (T0 + tj) + 2 * kq);
            nb = q + 1;
            for (int s = 0; s < NW && idx < total; ++s) advance();
          } else {
            pa[q] = pa[0]; pb[q] = pb[0]; pc[q] = pc[0];
          }
        }
#pragma unroll
        for (int q = 0; q < TB; ++q) c[q] = *pc[q];
#pragma unroll
        for (int ks = 0; ks < NB / 4; ++ks)
#pragma unroll
          for (int q = 0; q < TB; ++q) dmma884(c[q].x, c[q].y, -pa[q][4 * ks], pb[q][4 * ks]);
#pragma unroll
        for (int q = 0; q < TB; ++q)
          if (q < nb) *pc[q] = c[q];
      }
      __syncthreads();
    }
  }
  return true;
}

// Backward solves L' x = rhs for NRHS <= 2 right-hand sides held in shared memory (X + which * xs), panel by panel from
// the bottom: a half-warp per right-hand side walks the diagonal block, one thread per row above applies the panel.
template <int NT>
__device__ void blocked_backsolve(const Workspace& W, int p, double* X, int xs, int nrhs) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int LD = W.LD;
  const double* A = W.A;
  const int last = ((p - 1) / NB) * NB;
  for (int k0 = last; k0 >= 0; k0 -= NB) {
    const int nbk = min(NB, p - k0);
    if (warp == 0) {
      const int l = lane & 15, which = lane >> 4;
      const bool on = l < nbk && which < nrhs;
      double dl[NB];                                         // column l of the diagonal block: L[k0 + j][k0 + l], j > l
#pragma unroll
      for (int j = 0; j < NB; ++j) dl[j] = (on && j > l && j < nbk) ? A[(long long)(k0 + j) * LD + k0 + l] : 0.0;
      double x = on ? X[which * xs + k0 + l] : 0.0;
#pragma unroll
      for (int j = NB - 1; j >= 0; --j) {
        if (j < nbk) {
          const double xj = __shfl_sync(0xffffffffu, x, (lane & 16) | j) * W.sinv[k0 + j];
          if (l == j) x = xj;
          x = fma(-dl[j], xj, x);                            // dl[j] == 0 for j <= l
        }
      }
      if (on) X[which * xs + k0 + l] = x;
    }
    __syncthreads();
    if (k0 > 0) {
      for (int e = tid; e < nrhs * k0; e += NT) {
        const int which = e / k0, t = e - which * k0;
        const double* xb = X + which * xs + k0;
        double s = X[which * xs + t];
#pragma unroll 4
        for (int j = 0; j < nbk; ++j) s = fma(-A[(long long)(k0 + j) * LD + t], xb[j], s);
        X[which * xs + t] = s;
      }
      __syncthreads();
    }
  }
}

__device__ __forceinline__ Workspace carve(double* sm, double* global_A, int p, int n_extra, double** rest) {
  Workspace W;
  const int pp = (p + 15) & ~15;
  W.LD = pp + 4;
  W.rows_pad = (p + n_extra + 7) & ~7;
  double* q = sm;
  if (global_A) W.A = global_A;
  else { W.A = q; q += (long long)W.rows_pad * W.LD; }
  W.Pn = q; q += W.rows_pad * PLD;
  W.sD = q; q += NB * SDLD + 3;            // keep 16-byte alignment of what follows irrelevant: plain doubles
  W.sinv = q; q += pp;
  *rest = q;
  return W;
}

