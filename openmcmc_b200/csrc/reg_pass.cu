// reg_pass: the fused likelihood pass of the conjugate-regression hot path (SURVEY.md §8 a3/a4/a12).
//
// For every chain c, ONE streaming pass over (X_c, y_c [, w_c]) produces the sufficient statistics the
// NormalNormal / NormalGamma Gibbs updates need:
//     G   = X' W X          (p x p)   -- the reference's  (grad_param @ Q) @ grad_param.T,  location_scale.py:238-241
//     g   = X' W y          (p)       -- the reference's  A.T @ Q_rsp @ (y - d),            sampler.py:190-192
//     rss = (y-Xb)' W (y-Xb)          -- the reference's  residual.T @ P @ residual,        sampler.py:276,284
//     cnt = #(w > 0)                  -- the reference's  sum(P.diagonal() > 0),            sampler.py:283
// W = diag(w) (or I when w == nullptr); tau is NOT folded in here (ScaledMatrix scalar is applied by the consumers).
//
// reg_pass_kernel<PB, ..., SYRK>: one CTA (4 warps) per (chain, row split).  Rows are staged global -> shared by
// cp.async.bulk (TMA engine, one mbarrier per stage; 3 stages of 64 rows) into a chunked layout -- a stage is four
// contiguous chunks of 16 packed rows, chunk q shifted by 4 doubles, so that the four k-lanes of a DMMA fragment (one
// row from each chunk) read distinct banks; shapes or alignments the bulk path cannot take fall back to 16-byte
// cp.async (LDGSTS) into a padded row layout.  The SYRK runs on the FP64 tensor pipe: mma.sync.m8n8k4.f64 (SASS
// DMMA.8x8x4, the only native FP64 MMA shape on sm_100a).  A = X' and B = X come from the same tile, so one
// PB-register fragment set per 4 rows feeds all PB(PB+1)/2 lower-triangle 8x8 output tiles; at p = 64 every warp
// owns all 36 tiles (254 registers, 2 CTAs per SM) and the four warps split the rows.  g and rss ride on the FP64 FMA
// pipe (~5% of the DMMA work).  SYRK = false compiles the tensor work out: the explicit-residual stream (omc_reg_rss).
// 64 < p <= 512: gram_wide_kernel (64 x 64 panel pairs, a warp per 16 x 64 strip) + rss_wide_kernel below.
// With data-only weights both passes are PROLOGUE work: the sweep reads the record and the centre (DESIGN.md §3.1).
// Roofline (DESIGN.md): 46.1 MFLOP of DMMA per chain at n=10^4,p=64 vs 5.2 MB of HBM traffic => FP64-pipe bound.
#include "../../include/omc.h"
#include "omc_common.cuh"
#include "omc_internal.h"

namespace {

// measured best (profiles/r01_reg_pass_loader_variants.txt)
constexpr int KC = 64;             // rows per pipeline stage
constexpr int NSTAGE = 3;          // pipeline stages
constexpr int MINBLOCKS_WIDE = 2;  // CTAs per SM for the SYRK at PB >= 5 (every warp owns all tiles: 254 registers)
constexpr int NWARP = 4;
constexpr int NTHREADS = NWARP * 32;

struct RegPassArgs {
  const double* X;
  const double* y;
  const double* w;
  const double* beta;
  long long strideX, strideY, strideW, strideB;  // elements between consecutive chains (0 => shared by all chains)
  int n, p, n_chains, n_split, rows_per_split;
  double* out;  // records [chain][split][rec] ; rec = p*p + p + 2 : G | g | rss | cnt
};

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem, int src_bytes) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async8(void* smem, const void* gmem, int src_bytes) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(s), "l"(gmem), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

// ---- mbarrier + bulk async copy (TMA engine, SASS UBLKCP)
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

template <int PB>
struct Cfg {
  static constexpr int LD = 8 * PB + 4;  // padded row stride (doubles): (2g + 8k) mod 32 banks are distinct per phase
  static constexpr int STAGE_DOUBLES = KC * LD + 2 * KC;  // X tile | y | w
  static constexpr int NT = PB * (PB + 1) / 2;             // lower-triangle 8x8 tiles
  // chunked layout of the bulk path: a stage = 4 contiguous chunks of RC rows (one bulk copy each, rows packed at
  // stride 8*PB), chunk q shifted by 4 doubles so that the 4 k-lanes (one row from each chunk) hit distinct banks
  static constexpr int RC = KC / 4;
  static constexpr int CH = RC * 8 * PB + 4;
  static constexpr int RED_DOUBLES = NWARP * (NT * 64 + 8 * PB + 2);
  static constexpr int SMEM_DOUBLES = (NSTAGE * STAGE_DOUBLES > RED_DOUBLES) ? NSTAGE * STAGE_DOUBLES : RED_DOUBLES;
  static constexpr int BYTES = SMEM_DOUBLES * 8 + 64;  // + mbarriers
};

// SYRK = false: the residual-only pass (omc_reg_rss): no tensor work, no X'y; the same staging and fragment reads feed
// the per-row dot products only, so the pass is bound by the HBM stream of X.
template <int PB, bool WEIGHTED, bool SYRK = true>
struct Worker {
  using C = Cfg<PB>;
  double acc[C::NT][2];
  double gacc[PB];
  double bfrag[PB];
  double rss, cnt;
  int lane, g, kq;

  __device__ __forceinline__ void init(const RegPassArgs& a, int chain, int lane_) {
    lane = lane_;
    g = lane >> 2;
    kq = lane & 3;
#pragma unroll
    for (int t = 0; t < C::NT; ++t) acc[t][0] = acc[t][1] = 0.0;
#pragma unroll
    for (int jb = 0; jb < PB; ++jb) {
      gacc[jb] = 0.0;
      const int col = 8 * jb + g;  // per-lane slice of beta in fragment layout
      bfrag[jb] = (a.beta != nullptr && col < a.p) ? a.beta[(long long)chain * a.strideB + col] : 0.0;
    }
    rss = 0.0;
    cnt = 0.0;
  }

  // one stage = KC rows; warp w takes k-steps (4 rows each) w, w+NWARP, ...
  template <bool CHUNKED>
  __device__ __forceinline__ void stage(const double* Xs, int w) {
    constexpr int LD = C::LD;
    const double* ys = Xs + KC * LD;
    const double* ws = ys + KC;
#pragma unroll 2
    for (int ks = w; ks < KC / 4; ks += NWARP) {
      // padded layout: row 4ks+kq at stride LD ; chunked layout: row ks of chunk kq
      const int r = CHUNKED ? kq * C::RC + ks : 4 * ks + kq;
      const double* xr = CHUNKED ? Xs + kq * C::CH + ks * (8 * PB) + g : Xs + r * LD + g;
      double af[PB], bf[PB];
#pragma unroll
      for (int jb = 0; jb < PB; ++jb) af[jb] = xr[8 * jb];
      const double yv = ys[r];
      double wv = 1.0;
      if (WEIGHTED) {
        wv = ws[r];
#pragma unroll
        for (int jb = 0; jb < PB; ++jb) bf[jb] = af[jb] * wv;
      } else {
#pragma unroll
        for (int jb = 0; jb < PB; ++jb) bf[jb] = af[jb];
      }
      // SYRK tiles (lower triangle of the 8x8-block grid, row-major enumeration)
      if (SYRK) {
#pragma unroll
        for (int i = 0; i < PB; ++i)
#pragma unroll
          for (int j = 0; j <= i; ++j) {
            const int t = i * (i + 1) / 2 + j;
            // t < NT always holds; without the test the compiler lays out the PB = 1 kernels differently from the
            // measured build (profiles/r01_reg_pass_loader_variants.txt)
            if (t < C::NT) dmma884(acc[t][0], acc[t][1], af[i], bf[j]);
          }
#pragma unroll
        for (int jb = 0; jb < PB; ++jb) gacc[jb] = fma(bf[jb], yv, gacc[jb]);   // X' W y
      }
      {  // residual of the 4 rows of this k-step
        double dot = 0.0, dot1 = 0.0;   // two chains of fused multiply-adds (the residual-only pass has no DMMA to hide them)
#pragma unroll
        for (int jb = 0; jb < PB; jb += 2) {
          dot = fma(af[jb], bfrag[jb], dot);
          if (jb + 1 < PB) dot1 = fma(af[jb + 1], bfrag[jb + 1], dot1);
        }
        dot += dot1;
        dot += omc_shfl_xor(dot, 4);
        dot += omc_shfl_xor(dot, 8);
        dot += omc_shfl_xor(dot, 16);
        const double res = yv - dot;
        rss = fma(WEIGHTED ? wv * res : res, res, rss);
        if (WEIGHTED) cnt += (wv > 0.0) ? 1.0 : 0.0;
      }
    }
  }
};

// BULK = true : p == 8*PB and 16-byte aligned rows: 4 chunk copies + 1 y copy (+1 w) per stage through the TMA engine
//               (cp.async.bulk, completion on an mbarrier) -- no LSU traffic for staging, so the DMMA fragment LDS never
//               queue behind LDGSTS; the < KC-row tail is staged synchronously.
// BULK = false: generic cp.async (LDGSTS) path with zero-fill into the padded layout, any p / alignment.
template <int PB, bool WEIGHTED, bool BULK, bool SYRK>
__global__ void __launch_bounds__(NTHREADS, (PB > 4 && SYRK) ? MINBLOCKS_WIDE : 4) reg_pass_kernel(RegPassArgs a) {
  using C = Cfg<PB>;
  constexpr int LD = C::LD;
  extern __shared__ __align__(16) double smem[];

  const int chain = blockIdx.y, split = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int p = a.p, n = a.n;
  const int row0 = split * a.rows_per_split;
  const int row1 = min(n, row0 + a.rows_per_split);
  const int nrows = max(0, row1 - row0);
  const int nstage_total = (nrows + KC - 1) / KC;

  const double* Xc = a.X + (long long)chain * a.strideX + (long long)row0 * p;
  const double* yc = a.y + (long long)chain * a.strideY + row0;
  const double* wc = WEIGHTED ? a.w + (long long)chain * a.strideW + row0 : nullptr;

  // zero the staging area once: columns >= p of every row are never written by the loader and must read as 0
  for (int i = tid; i < NSTAGE * C::STAGE_DOUBLES; i += NTHREADS) smem[i] = 0.0;
  unsigned long long* full_bar = reinterpret_cast<unsigned long long*>(smem + C::SMEM_DOUBLES);
  if (BULK) {
    if (tid == 0) {
#pragma unroll
      for (int s = 0; s < NSTAGE; ++s) mbar_init(full_bar + s, 1);
      asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");  // generic zero-fill before async-proxy writes
  }
  __syncthreads();
  const int npipe = BULK ? nrows / KC : nstage_total;  // stages that go through the async pipeline

  const bool vec16 = ((p & 1) == 0) && ((((unsigned long long)Xc) & 15ull) == 0);
  const int fcpr = max(p >> 1, 1);                        // 16-byte chunks per row
  const bool fastrow = vec16 && (NTHREADS % fcpr == 0);   // thread -> fixed (row offset, chunk): no per-chunk division
  const int fr0 = tid / fcpr, fc0 = tid % fcpr, frstep = NTHREADS / fcpr;

  auto issue_stage = [&](int st) {
    if (BULK) {
      if (st < npipe && tid == 0) {
        double* Xs = smem + (st % NSTAGE) * C::STAGE_DOUBLES;
        double* ys = Xs + KC * LD;
        unsigned long long* bar = full_bar + (st % NSTAGE);
        const int r_base = st * KC;
        constexpr unsigned chunk_bytes = C::RC * 8 * PB * 8;
        mbar_expect_tx(bar, 4 * chunk_bytes + KC * 8u * (WEIGHTED ? 2u : 1u));
#pragma unroll
        for (int q = 0; q < 4; ++q)
          bulk_g2s(Xs + q * C::CH, Xc + (long long)(r_base + q * C::RC) * (8 * PB), chunk_bytes, bar);
        bulk_g2s(ys, yc + r_base, KC * 8u, bar);
        if (WEIGHTED) bulk_g2s(ys + KC, wc + r_base, KC * 8u, bar);
      }
      return;
    }
    if (st < nstage_total) {
      double* Xs = smem + (st % NSTAGE) * C::STAGE_DOUBLES;
      double* ys = Xs + KC * LD;
      double* ws = ys + KC;
      const int r_base = st * KC;
      const int valid = min(KC, nrows - r_base);
      const double* src = Xc + (long long)r_base * p;
      if (fastrow) {
        for (int r = fr0; r < KC; r += frstep) {
          const bool ok = r < valid;
          cp_async16(Xs + r * LD + 2 * fc0, ok ? (const void*)(src + (long long)r * p + 2 * fc0) : (const void*)Xc,
                     ok ? 16 : 0);
        }
      } else if (vec16) {
        const int total = KC * fcpr;
        for (int id = tid; id < total; id += NTHREADS) {
          const int r = id / fcpr, c = id - r * fcpr;
          const bool ok = r < valid;
          cp_async16(Xs + r * LD + 2 * c, ok ? (const void*)(src + (long long)r * p + 2 * c) : (const void*)Xc,
                     ok ? 16 : 0);
        }
      } else {
        const int total = KC * p;
        for (int id = tid; id < total; id += NTHREADS) {
          const int r = id / p, c = id - r * p;
          const bool ok = r < valid;
          cp_async8(Xs + r * LD + c, ok ? (const void*)(src + (long long)r * p + c) : (const void*)Xc, ok ? 8 : 0);
        }
      }
      for (int r = tid; r < KC; r += NTHREADS) {
        const bool ok = r < valid;
        cp_async8(ys + r, ok ? (const void*)(yc + r_base + r) : (const void*)yc, ok ? 8 : 0);
        if (WEIGHTED) cp_async8(ws + r, ok ? (const void*)(wc + r_base + r) : (const void*)wc, ok ? 8 : 0);
      }
    }
    cp_async_commit();
  };

  Worker<PB, WEIGHTED, SYRK> wk;
  wk.init(a, chain, lane);

#pragma unroll
  for (int s = 0; s < NSTAGE - 1; ++s) issue_stage(s);

  for (int st = 0; st < npipe; ++st) {
    if (BULK) {
      __syncthreads();  // buffer (st-1)%NSTAGE is free again
      issue_stage(st + NSTAGE - 1);
      mbar_wait(full_bar + (st % NSTAGE), (unsigned)((st / NSTAGE) & 1));
    } else {
      cp_async_wait<NSTAGE - 2>();
      __syncthreads();  // stage st has landed for everyone; buffer (st-1)%NSTAGE is free again
      issue_stage(st + NSTAGE - 1);
    }
    const double* Xs = smem + (st % NSTAGE) * C::STAGE_DOUBLES;
    wk.template stage<BULK>(Xs, warp);
  }
  if (!BULK) cp_async_wait<0>();
  __syncthreads();
  if (BULK && nrows - npipe * KC > 0) {
    // ragged tail (< KC rows): synchronous staging into buffer 0 (chunked layout), zero rows behind the data
    const int r_base = npipe * KC, valid = nrows - r_base;
    double* Xs = smem;
    double* ys = Xs + KC * LD;
    for (int id = tid; id < KC * 8 * PB; id += NTHREADS) {
      const int r = id / (8 * PB), c = id - r * (8 * PB);
      Xs[(r / C::RC) * C::CH + (r % C::RC) * (8 * PB) + c] = (r < valid) ? Xc[(long long)(r_base + r) * p + c] : 0.0;
    }
    for (int r = tid; r < KC; r += NTHREADS) {
      ys[r] = (r < valid) ? yc[r_base + r] : 0.0;
      if (WEIGHTED) ys[KC + r] = (r < valid) ? wc[r_base + r] : 0.0;
    }
    __syncthreads();
    wk.template stage<true>(Xs, warp);
    __syncthreads();
  }
  if (!SYRK) {
    // ---- residual-only pass: rss and cnt are the only outputs; G and g of the record stay as they are
    double r = (lane >> 2) == 0 ? wk.rss : 0.0, c = (lane >> 2) == 0 ? wk.cnt : 0.0;
    r = omc_warp_sum(r);
    c = omc_warp_sum(c);
    if (lane == 0) {
      smem[2 * warp] = r;
      smem[2 * warp + 1] = c;
    }
    __syncthreads();
    if (tid == 0) {
      double rs = 0.0, cs = 0.0;
      for (int q = 0; q < NWARP; ++q) {
        rs += smem[2 * q];
        cs += smem[2 * q + 1];
      }
      const int rec = p * p + p + 2;
      double* o = a.out + ((long long)chain * a.n_split + split) * rec;
      o[p * p + p] = rs;
      o[p * p + p + 1] = WEIGHTED ? cs : (double)nrows;
    }
    return;
  }

  // ---- combine the warps through shared memory (per warp: tiles | g | rss, cnt)
  constexpr int WREC = C::NT * 64 + 8 * PB + 2;
  double* red = smem + warp * WREC;
  const int g = lane >> 2, kq = lane & 3;
#pragma unroll
  for (int t = 0; t < C::NT; ++t) {
    red[t * 64 + 2 * lane] = wk.acc[t][0];
    red[t * 64 + 2 * lane + 1] = wk.acc[t][1];
  }
#pragma unroll
  for (int jb = 0; jb < PB; ++jb) {  // sum the 4 k-lanes
    double v = wk.gacc[jb];
    v += omc_shfl_xor(v, 1);
    v += omc_shfl_xor(v, 2);
    if (kq == 0) red[C::NT * 64 + 8 * jb + g] = v;
  }
  {
    // lanes sharing kq hold identical copies of each row's residual -> keep the g == 0 lanes only
    double r = (g == 0) ? wk.rss : 0.0, c = (g == 0) ? wk.cnt : 0.0;
    r = omc_warp_sum(r);
    c = omc_warp_sum(c);
    if (lane == 0) {
      red[C::NT * 64 + 8 * PB] = r;
      red[C::NT * 64 + 8 * PB + 1] = c;
    }
  }
  __syncthreads();

  if (warp == 0) {  // one writer warp sums the four warps
    const int rec = p * p + p + 2;
    double* o = a.out + ((long long)chain * a.n_split + split) * rec;
#pragma unroll
    for (int i = 0; i < PB; ++i)
#pragma unroll
      for (int j = 0; j <= i; ++j) {
        const int t = i * (i + 1) / 2 + j;
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          double v = 0.0;
          for (int q = 0; q < NWARP; ++q) v += smem[q * WREC + t * 64 + 2 * lane + e];
          const int rr = 8 * i + g, cc = 8 * j + 2 * kq + e;
          if (rr < p && cc < p) {
            o[rr * p + cc] = v;
            if (i != j) o[cc * p + rr] = v;
          }
        }
      }
    for (int c = lane; c < 8 * PB; c += 32) {
      double v = 0.0;
      for (int q = 0; q < NWARP; ++q) v += smem[q * WREC + C::NT * 64 + c];
      if (c < p) o[p * p + c] = v;
    }
    if (lane == 0) {
      double r = 0.0, c = 0.0;
      for (int q = 0; q < NWARP; ++q) {
        r += smem[q * WREC + C::NT * 64 + 8 * PB];
        c += smem[q * WREC + C::NT * 64 + 8 * PB + 1];
      }
      o[p * p + p] = r;
      o[p * p + p + 1] = WEIGHTED ? c : (double)nrows;
    }
  }
}

// sum the per-split records: out[c][e] = sum_s part[c][s][e] for the entries e >= e0 of a record
__global__ void reg_reduce_kernel(const double* part, double* out, int n_split, int rec, int e0, long long total) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int span = rec - e0;
  long long c = i / span;
  int e = e0 + (int)(i - c * span);
  const double* src = part + (c * n_split) * rec + e;
  double s = 0.0;
  for (int k = 0; k < n_split; ++k) s += src[(long long)k * rec];
  out[c * rec + e] = s;
}

template <int PB, bool W, bool B, bool SYRK>
int launch_one(const RegPassArgs& a, cudaStream_t st) {
  dim3 grid(a.n_split, a.n_chains);
  const int smem = Cfg<PB>::BYTES;
  OMC_CHECK_CUDA(cudaFuncSetAttribute(reg_pass_kernel<PB, W, B, SYRK>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  reg_pass_kernel<PB, W, B, SYRK><<<grid, NTHREADS, smem, st>>>(a);
  OMC_LAUNCH_CHECK();
  return 0;
}

template <int PB, bool SYRK>
int launch_pb(const RegPassArgs& a, bool weighted, cudaStream_t st) {
  // bulk (TMA-engine) copies need fully packed rows (p == 8*PB) and 16-byte aligned chunk starts for X, y and w
  auto al16 = [](const void* q) { return (((unsigned long long)q) & 15ull) == 0; };
  const bool bulk = (a.p == 8 * PB) && al16(a.X) && (a.strideX % 2 == 0) && al16(a.y) &&
                    (a.strideY % 2 == 0) && (!weighted || (al16(a.w) && (a.strideW % 2 == 0)));
  if (weighted) return bulk ? launch_one<PB, true, true, SYRK>(a, st) : launch_one<PB, true, false, SYRK>(a, st);
  return bulk ? launch_one<PB, false, true, SYRK>(a, st) : launch_one<PB, false, false, SYRK>(a, st);
}

template <bool SYRK>
int launch_any(const RegPassArgs& a, bool weighted, cudaStream_t st) {
  switch ((a.p + 7) / 8) {
    case 1: return launch_pb<1, SYRK>(a, weighted, st);
    case 2: return launch_pb<2, SYRK>(a, weighted, st);
    case 3: return launch_pb<3, SYRK>(a, weighted, st);
    case 4: return launch_pb<4, SYRK>(a, weighted, st);
    case 5: return launch_pb<5, SYRK>(a, weighted, st);
    case 6: return launch_pb<6, SYRK>(a, weighted, st);
    case 7: return launch_pb<7, SYRK>(a, weighted, st);
    default: return launch_pb<8, SYRK>(a, weighted, st);
  }
}


// ---------------------------------------------------------------------------------------------------------------
// p > 64: column panels.  G is built block by block: CTA (split, pair, chain) owns the 64 x 64 block (bi, bj), bi >= bj,
// of G = X'WX over its rows: A fragments from panel bi, B fragments from panel bj, all 64 8x8 tiles on the FP64 tensor
// pipe (DMMA.8x8x4); the pairs with bj == 0 also accumulate g = X'Wy for panel bi.  rss / cnt come from a separate
// streaming kernel (one warp per row, lanes over columns).  These run once per run (prologue) for models whose
// likelihood weights are data; staging is synchronous (no pipeline) -- the sweep itself never touches X (omc.h:
// omc_nn_dense_t.center).
constexpr int WK = 32;            // rows per stage
constexpr int WLD = 64 + 4;       // padded row stride of a staged panel
constexpr int WIDE_MAX_P = 512;

template <bool WEIGHTED>
__global__ void __launch_bounds__(NTHREADS) gram_wide_kernel(RegPassArgs a, int npan) {
  __shared__ __align__(16) double As[WK * WLD];
  __shared__ __align__(16) double Bs[WK * WLD];
  __shared__ double ys[WK], ws[WK];
  const int split = blockIdx.x, chain = blockIdx.z;
  int bi = 0, bj = 0;
  {  // pair index -> (bi, bj), bi >= bj
    int q = blockIdx.y;
    while (q > bi) { q -= bi + 1; ++bi; }
    bj = q;
  }
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, kq = lane & 3;
  const int p = a.p, n = a.n;
  const int row0 = split * a.rows_per_split, row1 = min(n, row0 + a.rows_per_split);
  const double* Xc = a.X + (long long)chain * a.strideX;
  const double* yc = a.y + (long long)chain * a.strideY;
  const double* wc = WEIGHTED ? a.w + (long long)chain * a.strideW : nullptr;
  const bool diag = bi == bj;
  const double* Bsm = diag ? As : Bs;
  // warp w owns the tile rows 2w, 2w+1 of the block (16 tiles, 64 accumulator registers) over ALL rows: no cross-warp sum
  double acc[16][2];
  double gacc[2];
#pragma unroll
  for (int t = 0; t < 16; ++t) acc[t][0] = acc[t][1] = 0.0;
  gacc[0] = gacc[1] = 0.0;
  for (int r0 = row0; r0 < row1; r0 += WK) {
    __syncthreads();
    for (int idx = tid; idx < WK * 64; idx += NTHREADS) {
      const int r = idx >> 6, c = idx & 63, row = r0 + r;
      const int ca = 64 * bi + c, cb = 64 * bj + c;
      const bool rok = row < row1;
      As[r * WLD + c] = (rok && ca < p) ? Xc[(long long)row * p + ca] : 0.0;
      if (!diag) Bs[r * WLD + c] = (rok && cb < p) ? Xc[(long long)row * p + cb] : 0.0;
    }
    for (int r = tid; r < WK; r += NTHREADS) {
      const int row = r0 + r;
      ys[r] = row < row1 ? yc[row] : 0.0;
      ws[r] = row < row1 ? (WEIGHTED ? wc[row] : 1.0) : 0.0;
    }
    __syncthreads();
#pragma unroll 2
    for (int ks = 0; ks < WK / 4; ++ks) {
      const int r = 4 * ks + kq;
      const double wv = ws[r], yv = ys[r];
      double af[2], bf[8];
      af[0] = As[r * WLD + 16 * warp + g];
      af[1] = As[r * WLD + 16 * warp + 8 + g];
#pragma unroll
      for (int j = 0; j < 8; ++j) bf[j] = Bsm[r * WLD + 8 * j + g] * wv;
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) dmma884(acc[i * 8 + j][0], acc[i * 8 + j][1], af[i], bf[j]);
      if (bj == 0) {
        gacc[0] = fma(af[0] * wv, yv, gacc[0]);
        gacc[1] = fma(af[1] * wv, yv, gacc[1]);
      }
    }
  }
  const int rec = p * p + p + 2;
  double* o = a.out + ((long long)chain * a.n_split + split) * rec;
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int rr = 64 * bi + 16 * warp + 8 * i + g, cc = 64 * bj + 8 * j + 2 * kq + e;
        if (rr < p && cc < p && (!diag || cc <= rr)) {
          const double v = acc[i * 8 + j][e];
          o[(long long)rr * p + cc] = v;
          if (rr != cc) o[(long long)cc * p + rr] = v;
        }
      }
  if (bj == 0) {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      double v = gacc[i];
      v += omc_shfl_xor(v, 1);
      v += omc_shfl_xor(v, 2);
      const int cc = 64 * bi + 16 * warp + 8 * i + g;
      if (kq == 0 && cc < p) o[(long long)p * p + cc] = v;
    }
  }
}

// rss = (y - X beta)' W (y - X beta) and cnt for any p: one warp per row, lanes over the columns (coalesced), beta in
// shared memory.  beta == NULL gives y'Wy.
template <bool WEIGHTED>
__global__ void __launch_bounds__(256) rss_wide_kernel(RegPassArgs a) {
  extern __shared__ double sbeta[];
  __shared__ double scratch[32];
  const int split = blockIdx.x, chain = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int p = a.p, n = a.n;
  const int row0 = split * a.rows_per_split, row1 = min(n, row0 + a.rows_per_split);
  for (int c = tid; c < p; c += 256) sbeta[c] = a.beta ? a.beta[(long long)chain * a.strideB + c] : 0.0;
  __syncthreads();
  const double* Xc = a.X + (long long)chain * a.strideX;
  const double* yc = a.y + (long long)chain * a.strideY;
  const double* wc = WEIGHTED ? a.w + (long long)chain * a.strideW : nullptr;
  double rss = 0.0, cnt = 0.0;
  for (int r = row0 + warp; r < row1; r += 16) {
    const int r2 = r + 8;
    const double* x1 = Xc + (long long)r * p;
    const double* x2 = Xc + (long long)r2 * p;
    const bool two = r2 < row1;
    double d1 = 0.0, d2 = 0.0;
    for (int c = lane; c < p; c += 32) {
      const double b = sbeta[c];
      d1 = fma(x1[c], b, d1);
      if (two) d2 = fma(x2[c], b, d2);
    }
    d1 = omc_warp_sum(d1);
    d2 = omc_warp_sum(d2);
    if (lane == 0) {
      const double w1 = WEIGHTED ? wc[r] : 1.0, e1 = yc[r] - d1;
      rss = fma(w1 * e1, e1, rss);
      cnt += (w1 > 0.0) ? 1.0 : 0.0;
      if (two) {
        const double w2 = WEIGHTED ? wc[r2] : 1.0, e2 = yc[r2] - d2;
        rss = fma(w2 * e2, e2, rss);
        cnt += (w2 > 0.0) ? 1.0 : 0.0;
      }
    }
  }
  rss = omc_block_sum(rss, scratch);
  cnt = omc_block_sum(cnt, scratch);
  if (tid == 0) {
    const int rec = p * p + p + 2;
    double* o = a.out + ((long long)chain * a.n_split + split) * rec;
    o[p * p + p] = rss;
    o[p * p + p + 1] = cnt;
  }
}

template <bool SYRK>
int launch_wide(const RegPassArgs& a, bool weighted, cudaStream_t st) {
  const int npan = (a.p + 63) / 64;
  if (SYRK) {
    dim3 grid(a.n_split, npan * (npan + 1) / 2, a.n_chains);
    if (weighted) gram_wide_kernel<true><<<grid, NTHREADS, 0, st>>>(a, npan);
    else gram_wide_kernel<false><<<grid, NTHREADS, 0, st>>>(a, npan);
    OMC_LAUNCH_CHECK();
  }
  dim3 grid2(a.n_split, a.n_chains);
  if (weighted) rss_wide_kernel<true><<<grid2, 256, a.p * sizeof(double), st>>>(a);
  else rss_wide_kernel<false><<<grid2, 256, a.p * sizeof(double), st>>>(a);
  OMC_LAUNCH_CHECK();
  return 0;
}

// Shared body of omc_reg_pass (SYRK = true) and omc_reg_rss (SYRK = false).
template <bool SYRK>
int reg_pass_impl(const double* X, long long strideX, const double* y, long long strideY, const double* w,
                  long long strideW, const double* beta, long long strideB, int n_chains, int n, int p, double* stats,
                  double* workspace, void* stream, const char* who) {
  int n_split = 1;
  long long ws = 0;
  int rc = omc_reg_pass_workspace(n_chains, n, p, &n_split, &ws);
  if (rc) return rc;
  OMC_REQUIRE(X && y && stats, "%s: null pointer", who);
  OMC_REQUIRE(SYRK || beta, "%s: beta missing", who);
  OMC_REQUIRE(n_split == 1 || workspace != nullptr, "%s: workspace required (n_split=%d)", who, n_split);
  OMC_REQUIRE(n_chains <= 65535, "%s: n_chains=%d exceeds grid.y; shard the chains", who, n_chains);
  cudaStream_t st = (cudaStream_t)stream;
  RegPassArgs a;
  a.X = X; a.y = y; a.w = w; a.beta = beta;
  a.strideX = strideX; a.strideY = strideY; a.strideW = strideW; a.strideB = strideB;
  a.n = n; a.p = p; a.n_chains = n_chains; a.n_split = n_split;
  int rps = (n + n_split - 1) / n_split;
  rps = ((rps + KC - 1) / KC) * KC;
  if (rps < KC) rps = KC;
  a.rows_per_split = rps;
  a.out = (n_split > 1) ? workspace : stats;
  if (p > 64) {
    OMC_REQUIRE(n_chains <= 65535, "%s: n_chains=%d exceeds the grid; shard the chains", who, n_chains);
    int rw = (n + n_split - 1) / n_split;
    a.rows_per_split = ((rw + WK - 1) / WK) * WK;
    rc = launch_wide<SYRK>(a, w != nullptr, st);
  } else {
    rc = launch_any<SYRK>(a, w != nullptr, st);
  }
  if (rc) return rc;
  if (n_split > 1) {
    const int rec = p * p + p + 2;
    const int e0 = SYRK ? 0 : p * p + p;   // the residual-only pass owns rss | cnt, G | g stay as they are
    long long total = (long long)n_chains * (rec - e0);
    reg_reduce_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(workspace, stats, n_split, rec, e0, total);
    OMC_LAUNCH_CHECK();
  }
  return 0;
}

}  // namespace

extern "C" int omc_reg_pass_workspace(int n_chains, int n, int p, int* n_split_out, long long* workspace_doubles) {
  OMC_REQUIRE(n_chains > 0 && n >= 0 && p > 0, "omc_reg_pass_workspace: bad shape C=%d n=%d p=%d", n_chains, n, p);
  OMC_REQUIRE(p <= WIDE_MAX_P, "omc_reg_pass: p=%d > %d is not supported", p, WIDE_MAX_P);
  int sms = omc_sm_count();
  int max_split = (n + KC - 1) / KC;
  if (max_split < 1) max_split = 1;
  long long ctas_per_split = n_chains;              // p > 64: one CTA per (chain, 64-column panel pair)
  if (p > 64) ctas_per_split *= ((p + 63) / 64) * (((p + 63) / 64) + 1) / 2;
  int want = (int)((4ll * sms + ctas_per_split - 1) / ctas_per_split);  // aim for >= 4 CTAs per SM when chains are few
  int s = want < 1 ? 1 : (want > max_split ? max_split : want);
  *n_split_out = s;
  *workspace_doubles = (s > 1) ? (long long)n_chains * s * ((long long)p * p + p + 2) : 0;
  return 0;
}

extern "C" int omc_reg_pass(const double* X, long long strideX, const double* y, long long strideY, const double* w,
                            long long strideW, const double* beta, long long strideB, int n_chains, int n, int p,
                            double* stats, double* workspace, void* stream) {
  return reg_pass_impl<true>(X, strideX, y, strideY, w, strideW, beta, strideB, n_chains, n, p, stats, workspace, stream,
                             "omc_reg_pass");
}

// Residual-only pass: rss = (y - X beta)' W (y - X beta) and cnt into the record, G and g untouched (they depend on the
// data alone; the sweep plan keeps them from the prologue's omc_reg_pass).  ref: sampler.py:276,283-284
extern "C" int omc_reg_rss(const double* X, long long strideX, const double* y, long long strideY, const double* w,
                           long long strideW, const double* beta, long long strideB, int n_chains, int n, int p,
                           double* stats, double* workspace, void* stream) {
  return reg_pass_impl<false>(X, strideX, y, strideY, w, strideW, beta, strideB, n_chains, n, p, stats, workspace, stream,
                              "omc_reg_rss");
}
