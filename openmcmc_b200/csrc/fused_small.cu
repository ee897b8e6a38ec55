// omc_fused_small: a list of per-chain O(1) / O(p) operations in one launch (include/omc.h).  The arithmetic of every op
// is that of its stand-alone kernel (logp.cu, dense_draw.cu, omc_api.cu); sums over the elements of one chain run in
// element order here (one thread per chain) instead of the stand-alone kernels' block reductions.
//   ref: mcmc.py:105-111 (store epilogue), sampler.py:252-288 (NormalGamma), distribution.py:241-261, 490-508,
//        location_scale.py:145-167 (log-densities)
#include "../../include/omc.h"
#include "omc_common.cuh"
#include "omc_internal.h"

namespace {
constexpr int FS_THREADS = 128;
constexpr double LOG_2PI = 1.8378770664093454835606594728112;

__device__ __forceinline__ double fvat(const omc_vec_t& v, int chain, long long i, double dflt) {
  return v.ptr ? v.ptr[(long long)chain * v.chain_stride + i] : dflt;
}

__device__ __forceinline__ void op_normal_ss(const omc_logp_normal_ss_t& a, int c) {
  const double s = fvat(a.scalar, c, 0, 1.0);
  const double v = 0.5 * (a.dim * log(s) + fvat(a.logdet, c, 0, 0.0) - a.dim * LOG_2PI - s * fvat(a.ss, c, 0, 0.0));
  a.out[c] = a.accumulate ? a.out[c] + v : v;
}
// LPC lanes per chain (1 or 32): element loops are strided over the lanes and summed by a shuffle tree, everything
// that is one value per chain is done by lane 0 of the chain.
template <int LPC>
__device__ __forceinline__ double lanes_sum(double v) { return LPC == 32 ? omc_warp_sum(v) : v; }

template <int LPC>
__device__ __forceinline__ void op_gamma(const omc_logp_gamma_t& a, int c, int l) {
  double acc = 0.0;
  for (int i = l; i < a.n_elem; i += LPC) {
    const double x = fvat(a.x, c, i, 0.0);
    const double sh = fvat(a.shape, c, a.shape_len > 1 ? i : 0, 1.0);
    const double rt = fvat(a.rate, c, a.rate_len > 1 ? i : 0, 1.0);
    const double scale = 1.0 / rt;
    const double y = x / scale;
    double lp = omc_xlogy(sh - 1.0, y) - y - lgamma(sh) - log(scale);
    if (!(sh > 0.0) || rt < 0.0) lp = nan("");               // scipy: invalid shape / rate -> nan
    else if (!(y >= 0.0)) lp = isnan(y) ? y : -INFINITY;
    acc += lp;
  }
  acc = lanes_sum<LPC>(acc);
  if (l == 0) a.out[c] = a.accumulate ? a.out[c] + acc : acc;
}
template <int LPC>
__device__ __forceinline__ void op_poisson(const omc_logp_poisson_t& a, int c, int l) {
  double acc = 0.0;
  for (int i = l; i < a.n_elem; i += LPC) {
    const double k = fvat(a.k, c, i, 0.0);
    const double mu = fvat(a.rate, c, a.rate_len > 1 ? i : 0, 1.0);
    double lp = omc_xlogy(k, mu) - lgamma(k + 1.0) - mu;
    if (!(mu >= 0.0)) lp = nan("");                           // scipy: invalid rate -> nan
    else if (!(k >= 0.0) || floor(k) != k) lp = isnan(k) ? k : -INFINITY;   // off the support
    acc += lp;
  }
  acc = lanes_sum<LPC>(acc);
  if (l == 0) a.out[c] = a.accumulate ? a.out[c] + acc : acc;
}
template <int LPC>
__device__ __forceinline__ void op_ng_draw(const omc_ng_draw_t& a, int c, int l) {
  const int ne = a.n_elem > 0 ? a.n_elem : 1;
  OmcRng rng;
  rng.seed = a.rng.seed; rng.sweep = a.rng.sweep; rng.chain_offset = a.rng.chain_offset; rng.site = a.rng.site;
  for (int k = l; k < ne; k += LPC) {
    const long long t = (long long)c * ne + k;
    const double shape = fvat(a.a0, c, a.a0_len > 1 ? k : 0, 0.0) + 0.5 * fvat(a.cnt, c, k * a.cnt_stride, 0.0);
    const double rate = fvat(a.b0, c, a.b0_len > 1 ? k : 0, 0.0) + 0.5 * fvat(a.ss, c, k * a.ss_stride, 0.0);
    if (a.probe_a) a.probe_a[t] = shape;
    if (a.probe_b) a.probe_b[t] = rate;
    double gvar;
    if (a.debug_g) gvar = a.debug_g[(a.rng.sweep ? (long long)(*a.rng.sweep) : 0ll) * a.debug_sweep_stride + t];
    else gvar = omc_std_gamma(rng, c, (unsigned int)k << 12, shape);
    a.out[t] = (rate == 0.0) ? INFINITY : gvar * (1.0 / rate);   // reference: scale = inf when rate == 0 (sampler.py:285-286)
  }
}
template <int LPC>
__device__ __forceinline__ void op_quadform(const omc_quadform_t& a, int c, int l) {   // scaled identity / diagonal P only
  double ss = 0.0, cnt = 0.0;
  for (int i = l; i < a.p; i += LPC) {                        // (the stand-alone kernel's order at LPC = 32)
    const double ri = fvat(a.x, c, i, 0.0) - fvat(a.mu, c, i, 0.0);
    const double d = a.kind == OMC_MAT_DIAG ? a.P.ptr[(long long)c * a.P.chain_stride + i]
                                            : (a.P.ptr ? a.P.ptr[(long long)c * a.P.chain_stride] : 1.0);
    ss += d * ri * ri;
    cnt += (d > 0.0) ? 1.0 : 0.0;
  }
  ss = lanes_sum<LPC>(ss);
  cnt = lanes_sum<LPC>(cnt);
  if (l == 0) {
    a.ss[c] = ss;
    a.cnt[c] = cnt;
  }
}

// 7 CTAs per SM (<= 72 registers): the 1024 CTAs of 4096 chains at 32 lanes per chain run in one wave on 148 SMs
// (6 at the 80 registers the compiler picks unbounded: 1.15 waves)
template <int LPC>
__global__ void __launch_bounds__(FS_THREADS, 7) fused_small_kernel(const __grid_constant__ omc_fused_small_t a) {
  const long long gtid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long nthreads = (long long)gridDim.x * blockDim.x;
  const long long chain_ll = gtid / LPC;
  const int c = (int)chain_ll, l = (int)(gtid % LPC);
  const bool live = chain_ll < a.n_chains;                  // warp-uniform at LPC = 32
  for (int q = 0; q < a.n_ops; ++q) {
    const omc_fop_t& op = a.ops[q];
    if (q && LPC > 1) __syncwarp();                           // lane 0 wrote what the other lanes of the chain read next
    switch (op.kind) {
      case OMC_FOP_LOGP_NORMAL_SS: if (live && l == 0) op_normal_ss(op.u.normal_ss, c); break;
      case OMC_FOP_LOGP_GAMMA: if (live) op_gamma<LPC>(op.u.gamma, c, l); break;
      case OMC_FOP_LOGP_POISSON: if (live) op_poisson<LPC>(op.u.poisson, c, l); break;
      case OMC_FOP_LOGP_CONST:
        if (live && l == 0) op.u.konst.out[c] = op.u.konst.accumulate ? op.u.konst.out[c] + op.u.konst.value : op.u.konst.value;
        break;
      case OMC_FOP_NG_DRAW: if (live) op_ng_draw<LPC>(op.u.ng, c, l); break;
      case OMC_FOP_QUADFORM: if (live) op_quadform<LPC>(op.u.quad, c, l); break;
      case OMC_FOP_STORE_COPY: {
        unsigned long long it = *op.u.copy.iter_counter;
        if (op.u.copy.ring) it %= (unsigned long long)op.u.copy.max_iter;
        else if ((long long)it >= op.u.copy.max_iter) break;
        double* d = op.u.copy.dst + it * op.u.copy.count;
        if (op.u.copy.count == a.n_chains) {                  // one value per chain (maybe produced above): its own lane 0
          if (live && l == 0) d[c] = op.u.copy.src[c];
        } else {
          for (long long i = gtid; i < op.u.copy.count; i += nthreads) d[i] = op.u.copy.src[i];
        }
        break;
      }
      default: break;
    }
  }
}
}  // namespace

extern "C" int omc_fused_small(const omc_fused_small_t* a, void* stream) {
  OMC_REQUIRE(a && a->n_chains >= 1 && a->n_ops >= 1 && a->n_ops <= OMC_FUSED_MAX_OPS, "omc_fused_small: bad argument");
  for (int q = 0; q < a->n_ops; ++q) {
    const omc_fop_t& op = a->ops[q];
    OMC_REQUIRE(op.kind >= OMC_FOP_LOGP_NORMAL_SS && op.kind <= OMC_FOP_STORE_COPY, "omc_fused_small: op %d has kind %d", q, op.kind);
    if (op.kind == OMC_FOP_QUADFORM)
      OMC_REQUIRE(op.u.quad.kind == OMC_MAT_EYE || (op.u.quad.kind == OMC_MAT_DIAG && op.u.quad.P.ptr),
                  "omc_fused_small: op %d: only scaled-identity / diagonal quadratic forms are fused", q);
    if (op.kind == OMC_FOP_STORE_COPY) {
      OMC_REQUIRE(op.u.copy.src && op.u.copy.dst && op.u.copy.iter_counter && op.u.copy.max_iter >= 1, "omc_fused_small: op %d: bad copy", q);
      for (int e = 0; e < q; ++e) {       // a source produced inside this launch: only the per-chain layout is safe
        const omc_fop_t& pe = a->ops[e];
        const double* out = pe.kind == OMC_FOP_LOGP_NORMAL_SS ? pe.u.normal_ss.out : pe.kind == OMC_FOP_LOGP_GAMMA ? pe.u.gamma.out
                          : pe.kind == OMC_FOP_LOGP_POISSON ? pe.u.poisson.out : pe.kind == OMC_FOP_LOGP_CONST ? pe.u.konst.out
                          : pe.kind == OMC_FOP_NG_DRAW ? pe.u.ng.out : pe.kind == OMC_FOP_QUADFORM ? pe.u.quad.ss : nullptr;
        if (out && out == op.u.copy.src)
          OMC_REQUIRE(op.u.copy.count == a->n_chains, "omc_fused_small: op %d copies %lld values produced by op %d of the same launch", q, op.u.copy.count, e);
      }
    }
  }
  // lanes per chain: a warp when some op loops over more than a few elements per chain (C4: 32 Poisson / Gamma terms,
  // C2: a 64-term quadratic form), one thread otherwise; store copies are spread over the whole grid, so it grows with
  // the largest copy (<= 2 CTAs per SM)
  int widest = 1;
  for (int q = 0; q < a->n_ops; ++q) {
    const omc_fop_t& op = a->ops[q];
    const int w = op.kind == OMC_FOP_LOGP_GAMMA ? op.u.gamma.n_elem : op.kind == OMC_FOP_LOGP_POISSON ? op.u.poisson.n_elem
                : op.kind == OMC_FOP_QUADFORM ? op.u.quad.p : op.kind == OMC_FOP_NG_DRAW ? op.u.ng.n_elem : 1;
    if (w > widest) widest = w;
  }
  const int lpc = widest > 4 ? 32 : 1;
  long long grid_ll = ((long long)a->n_chains * lpc + FS_THREADS - 1) / FS_THREADS;
  for (int q = 0; q < a->n_ops; ++q)
    if (a->ops[q].kind == OMC_FOP_STORE_COPY) {
      long long want = (a->ops[q].u.copy.count + 8 * FS_THREADS - 1) / (8 * FS_THREADS);
      const long long cap = 2ll * omc_sm_count();
      if (want > cap) want = cap;
      if (want > grid_ll) grid_ll = want;
    }
  const unsigned grid = (unsigned)grid_ll;
  if (lpc == 32) fused_small_kernel<32><<<grid, FS_THREADS, 0, (cudaStream_t)stream>>>(*a);
  else fused_small_kernel<1><<<grid, FS_THREADS, 0, (cudaStream_t)stream>>>(*a);
  OMC_LAUNCH_CHECK();
  return 0;
}
