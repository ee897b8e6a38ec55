// Truncated-prior NormalNormal draw for 64 < p <= 512 (SURVEY.md §8 f3): ONE coordinate-wise Gibbs scan from the current
// beta, the same computation as nn_truncated_scan_kernel (dense_draw.cu), which keeps Q in shared memory up to p = 64:
//   Q = lam*P0 + tau*G,  b = lam*P0 mu0 + tau*g,
//   beta_i ~ N(v_i (b_i - sum_{j != i} Q_ij beta_j), v_i = 1/Q_ii) truncated to [lo_i, hi_i],  i = 0 .. p-1
// with one uniform per coordinate (Philox block i of the chain, or debug_u) behind the truncnorm inverse CDF.
//   ref: sampler.py:196-205, gmrf.py:201-266
//
// Q does not fit in shared memory here (2 MB per chain at p = 512) and the scan is sequential over coordinates, so:
//   - one warp per chain, several independent warps per CTA and no CTA barrier: throughput comes from chains in flight;
//   - the rows of G (and of P0 when it is dense) are streamed in order through a two-slot per-warp ring in shared
//     memory, 1-D bulk copies (TMA engine) completing on one mbarrier per slot, with an L2 prefetch PF_AHEAD rows ahead;
//     a row that starts at an odd double is copied as its 16-byte aligned envelope (one extra double in front), and an
//     element the envelope cannot cover without leaving the array is read with a plain load;
//   - beta lives in registers, element j = s*32 + lane in x[s] of lane j % 32;
//   - the reduction is off the dependent path: while step i draws x_i, the warp sums row i+1 against every coordinate
//     except i and i+1 (S), and takes Q_{i+1,i}, Q_{i+1,i+1}, b_{i+1}, the bounds and the uniform of coordinate i+1;
//     after the draw only  r = b - (S + Q_{i+1,i} x_i)  remains, then the truncnorm, which every lane evaluates with
//     the same operands (no broadcast).
#include "../../include/omc.h"
#include "omc_common.cuh"
#include "omc_internal.h"
#include "omc_special.cuh"

namespace {

constexpr int TS_WARPS = 4;    // warps (chains) per CTA
constexpr int TS_SLOTS = 2;    // ring slots per warp: row i+1 in use while row i+2 arrives
constexpr int PF_AHEAD = 6;    // rows between the L2 prefetch and the bulk copy into the ring

__device__ __forceinline__ unsigned smem_addr(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_addr(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
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
      "}\n" ::"r"(smem_addr(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                   smem_addr(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(smem_addr(bar))
               : "memory");
}
// L2 prefetch of the 16-byte granules of src[-1, n) that lie wholly inside it (a row r >= 1: the double in front of it
// belongs to row r - 1)
__device__ __forceinline__ void prefetch_l2(const double* src, int n) {
  const unsigned long long a = (unsigned long long)src & ~15ull;
  const unsigned bytes = (unsigned)(((unsigned long long)(src + n) & ~15ull) - a);
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;\n" ::"l"(a), "r"(bytes) : "memory");
}

__device__ __forceinline__ double vec_at(const omc_vec_t& v, int chain, int i, double dflt) {
  return v.ptr ? v.ptr[(long long)chain * v.chain_stride + i] : dflt;
}

// Row src[0, n) of an array that spans [base, limit) into dst (16-byte aligned), element j at dst[shift + j] with
// shift = 1 when src is not 16-byte aligned.  Lane 0 only.  The aligned envelope goes out as one bulk copy; an end
// element whose envelope would leave [base, limit) is stored from a plain load instead (the other lanes read the row
// after a __syncwarp that follows this store).  issue = false: only the bytes the bulk copy will bring.
__device__ __forceinline__ unsigned stage_row(double* dst, const double* src, int n, const double* base,
                                              const double* limit, unsigned long long* bar, bool issue) {
  const double* lo = reinterpret_cast<const double*>((unsigned long long)src & ~15ull);
  const double* hi = reinterpret_cast<const double*>(((unsigned long long)(src + n) + 15ull) & ~15ull);
  const double* b0 = lo < base ? lo + 2 : lo;
  const double* b1 = hi > limit ? hi - 2 : hi;
  if (!issue) return (unsigned)((b1 - b0) * 8);
  if (b0 != lo) dst[1] = src[0];
  if (b1 != hi) dst[(src - lo) + n - 1] = src[n - 1];
  bulk_g2s(dst + (b0 - lo), b0, (unsigned)((b1 - b0) * 8), bar);
  return 0;
}

template <int NS>
__global__ void __launch_bounds__(TS_WARPS * 32, 3) nn_trunc_stream_kernel(omc_nn_dense_t a) {
  extern __shared__ __align__(16) unsigned char ts_sm[];
  const int p = a.p, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int chain = blockIdx.x * TS_WARPS + wid;
  if (chain >= a.n_chains) return;
  const bool dense = a.prior_kind == OMC_MAT_DENSE;
  const int ld = (p + 2) & ~1;                     // slot row stride (doubles): a row plus its envelope, 16-byte rows
  const int rows = dense ? 2 : 1;                  // G row, then P0 row
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(ts_sm) + wid * TS_SLOTS;
  double* ring = reinterpret_cast<double*>(ts_sm + 16 * TS_WARPS) + (long long)wid * TS_SLOTS * rows * ld;

  const double* rec = a.stats.ptr + (long long)chain * a.stats.chain_stride;
  const double* P0 = dense ? a.prior_P.ptr + (long long)chain * a.prior_P.chain_stride : nullptr;
  const double tau = vec_at(a.tau, chain, 0, 1.0);
  const double lam = vec_at(a.lambda, chain, 0, 1.0);
  // the arrays the envelopes must stay inside: this chain's record (G | g | rss | cnt), this chain's P0
  const double* rec_end = rec + (long long)p * p + p + 2;
  const double* P0_end = dense ? P0 + (long long)p * p : nullptr;

  if (lane == 0) {
    for (int s = 0; s < TS_SLOTS; ++s) mbar_init(&bars[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  __syncwarp();
  // row r into slot r % TS_SLOTS (lane 0)
  auto fill = [&](int r) {
    double* slot = ring + (r % TS_SLOTS) * rows * ld;
    unsigned long long* bar = &bars[r % TS_SLOTS];
    const double* g = rec + (long long)r * p;
    unsigned bytes = stage_row(slot, g, p, rec, rec_end, bar, false);
    if (dense) bytes += stage_row(slot + ld, P0 + (long long)r * p, p, P0, P0_end, bar, false);
    mbar_expect_tx(bar, bytes);   // before the copies: the transaction count cannot complete the phase early
    stage_row(slot, g, p, rec, rec_end, bar, true);
    if (dense) stage_row(slot + ld, P0 + (long long)r * p, p, P0, P0_end, bar, true);
    const int rp = r + PF_AHEAD;
    if (rp < p) {
      prefetch_l2(rec + (long long)rp * p, p);
      if (dense) prefetch_l2(P0 + (long long)rp * p, p);
    }
  };
  if (lane == 0) {
    for (int r = 1; r < PF_AHEAD && r < p; ++r) {
      prefetch_l2(rec + (long long)r * p, p);
      if (dense) prefetch_l2(P0 + (long long)r * p, p);
    }
    fill(0);
    fill(1);
  }
  __syncwarp();                                    // lane 0's plain-load elements of rows 0 and 1

  double* bt = a.beta + (long long)chain * p;
  double x[NS];
#pragma unroll
  for (int s = 0; s < NS; ++s) x[s] = (s * 32 + lane < p) ? bt[s * 32 + lane] : 0.0;
  const double* du = a.debug_u ? a.debug_u + (a.rng.sweep ? (long long)(*a.rng.sweep) : 0ll) * a.debug_sweep_stride +
                                     (long long)chain * p
                               : nullptr;
  OmcRng rng;
  rng.seed = a.rng.seed; rng.sweep = a.rng.sweep; rng.chain_offset = a.rng.chain_offset; rng.site = a.rng.site;
  const double* mu0 = a.mu0.ptr ? a.mu0.ptr + (long long)chain * a.mu0.chain_stride : nullptr;
  const double p0_eye = a.prior_P.ptr ? a.prior_P.ptr[(long long)chain * a.prior_P.chain_stride] : 1.0;

  // Everything coordinate k needs that does not depend on x_{k-1}: S = sum_{j != k-1, k} Q_kj x_j, c = Q_{k,k-1},
  // q = Q_kk, b_k, bounds, uniform; taken from row k at the top of step k - 1 of the loop below.
  double nS = 0.0, nc = 0.0, nq = 0.0, nb = 0.0, nlo = 0.0, nhi = 0.0, nu = 0.0;
  bool bad = false;

  double xprev = 0.0;
  for (int i = -1; i < p; ++i) {                   // i = -1: the terms of coordinate 0 only
    const double S = nS, c = nc, q = nq, bi = nb, lo = nlo, hi = nhi, u = nu;
    __syncwarp();                                   // every lane is done with row i: its slot takes row i + 2
    if (lane == 0 && i >= 0 && i + 2 < p) fill(i + 2);
    if (i + 1 < p) {                                // excludes x_i (old) and x_{i+1}: independent of this draw
      const int k = i + 1;
      mbar_wait(&bars[k % TS_SLOTS], (unsigned)((k / TS_SLOTS) & 1));
      const double* slot = ring + (k % TS_SLOTS) * rows * ld;
      const int gsh = (int)(((unsigned long long)(rec + (long long)k * p) >> 3) & 1);
      const double* grow = slot + gsh;
      const double* prow = dense ? slot + ld + (int)(((unsigned long long)(P0 + (long long)k * p) >> 3) & 1) : nullptr;
      double pkk;                                      // P0_kk
      if (dense) pkk = prow[k];
      else if (a.prior_kind == OMC_MAT_DIAG) pkk = a.prior_P.ptr[(long long)chain * a.prior_P.chain_stride + k];
      else pkk = p0_eye;
      double sx = 0.0, sm = 0.0;
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        const int j = s * 32 + lane;
        if (j < p) {
          double qj = tau * grow[j];
          if (dense) {
            const double pk = prow[j];
            qj = lam * pk + qj;
            if (mu0) sm = fma(lam * pk, mu0[j], sm);
          }
          if (j != k && j != k - 1) sx = fma(qj, x[s], sx);
          if (a.probe_Q) a.probe_Q[(long long)chain * p * p + (long long)k * p + j] = (!dense && j == k) ? lam * pkk + qj : qj;
        }
      }
      sx = omc_warp_sum(sx);
      if (dense) sm = omc_warp_sum(sm);
      nq = lam * pkk + tau * grow[k];
      nc = 0.0;
      if (k > 0) nc = dense ? lam * prow[k - 1] + tau * grow[k - 1] : tau * grow[k - 1];
      nS = sx;
      if (!dense) sm = mu0 ? lam * pkk * mu0[k] : 0.0;
      nb = sm + tau * rec[(long long)p * p + k];
      nlo = a.trunc_lo.ptr ? vec_at(a.trunc_lo, chain, a.trunc_lo_len > 1 ? k : 0, 0.0) : -INFINITY;
      nhi = a.trunc_hi.ptr ? vec_at(a.trunc_hi, chain, a.trunc_hi_len > 1 ? k : 0, 0.0) : INFINITY;
      if (du) nu = du[k];
      else {
        const uint4 blk = omc_rng_block(rng, chain, (unsigned int)k);
        nu = omc_u01(blk.x, blk.y);
      }
      if (a.probe_b && lane == 0) a.probe_b[(long long)chain * p + k] = nb;
    }
    if (i < 0) continue;
    const double v = 1.0 / q;
    const double mean = v * (bi - fma(c, xprev, S));
    const double xn = omc_truncated_normal_rv(mean, sqrt(v), lo, hi, u);
    bad |= !(q > 0.0);
    const int si = lane == (i & 31) ? i >> 5 : -1;
#pragma unroll
    for (int s = 0; s < NS; ++s) x[s] = s == si ? xn : x[s];
    xprev = xn;                                     // enters coordinate i+1 through c, the later ones through x[]
  }
#pragma unroll
  for (int s = 0; s < NS; ++s)
    if (s * 32 + lane < p) bt[s * 32 + lane] = x[s];
  if (lane == 0 && bad && a.status) atomicOr(&a.status[chain], OMC_STATUS_NOT_PD);
}

template <int NS>
int launch(const omc_nn_dense_t& a, cudaStream_t st) {
  const int ld = (a.p + 2) & ~1, rows = a.prior_kind == OMC_MAT_DENSE ? 2 : 1;
  const size_t smem = 16 * TS_WARPS + (size_t)TS_WARPS * TS_SLOTS * rows * ld * sizeof(double);
  OMC_CHECK_CUDA(cudaFuncSetAttribute(nn_trunc_stream_kernel<NS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  nn_trunc_stream_kernel<NS><<<(a.n_chains + TS_WARPS - 1) / TS_WARPS, TS_WARPS * 32, smem, st>>>(a);
  OMC_LAUNCH_CHECK();
  return 0;
}

}  // namespace

int omc_launch_trunc_stream(const omc_nn_dense_t& a, cudaStream_t st) {
  if (a.p <= 128) return launch<4>(a, st);
  if (a.p <= 256) return launch<8>(a, st);
  return launch<16>(a, st);
}
