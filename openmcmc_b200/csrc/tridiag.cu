// Temporal-GMRF NormalNormal draw with a TRIDIAGONAL posterior precision (SURVEY.md §8 a3, a7-a11; BASELINE configs[2]).
//
//   Q = lambda*P + tau*W  (P tridiagonal RW1 precision shared by all chains, W diagonal or identity)
//   b = lambda*P*mu0 + tau*W*y ;  L = chol(Q) in natural order ;  x = L^-T (L^-1 b + z)
//   ref: sampler.py:154-207 (NormalNormal.sample), gmrf.py:167-198 (sample_normal_canonical), gmrf.py:489-520
//        (sparse_cholesky: SuperLU, natural ordering, no pivoting == the Thomas-order recurrence), gmrf.py:437-462, 29-61
//
// LDL' form (L = L~ D^1/2, so x = L~^-T (D^-1 L~^-1 b + D^-1/2 z) is the reference's mu + L^-T z exactly):
//   pivots    u_i = d_i - e_{i-1}^2 / u_{i-1}
//   forward   f_i = b_i - m_{i-1} f_{i-1},          m_i = e_i / u_i
//   draw      g_i = f_i / u_i + z_i / sqrt(u_i)
//   backward  x_i = g_i - m_i x_{i+1}
// The reference runs these sequentially (1e6 dependent steps per chain).  Here a tile is 128 threads x 18 consecutive
// elements, and three kernels do the work with ONE read of y each and no per-element scratch in HBM:
//
//  tg_aggregate_kernel pivots and forward solve as ONE projective linear recurrence on s_i = (p_i, p_{i-1}, h_i),
//                      u_i = p_i/p_{i-1}, f_i = h_i/p_{i-1}:   p_i = d_i p_{i-1} - e_{i-1}^2 p_{i-2},
//                      h_i = b_i p_{i-1} - e_{i-1} h_{i-1}.  Element maps compose as 3x3 block-triangular matrices (7
//                      entries, no divisions); thread aggregates -> CTA scan.  Pure streaming: writes every thread's
//                      exclusive prefix inside its tile (56 B per 18 elements) and the tile total.
//  tg_tilescan_kernel  one CTA per chain scans the tile totals -> the exact (u, f) entering every tile.
//  tg_solve_kernel     draws the tile's normals (four per Philox block, fp32 special-function unit for the
//                      transcendental parts) while its TMA loads are in flight, forms the exact (1/u, f) entering each
//                      thread's 18 elements, re-runs the *sequential* recurrences on them (so every pivot / f / g comes
//                      from the reference's operation sequence), keeps g and m in registers, builds the backward affine
//                      aggregate on the way, scans it (CTA + reverse decoupled look-back over tiles), then walks back
//                      down producing x and both quadratic forms (x-mu0)'P(x-mu0), (y-x)'W(y-x) in the same pass.
//                      x leaves through shared memory with one bulk (TMA-engine) store per tile.
//
// Tiles are staged global -> shared with cp.async.bulk (1-D, completion on an mbarrier); a thread's 18 elements sit at a
// 144-byte stride, so 16-byte LDS/STS are bank-conflict free.  Work is tile-major (tile t of all chains, then t+1): the
// chains read the same tile of the shared P together (L2), and in the solve kernel an atomic ticket guarantees that the
// tiles a look-back waits on are running or done.  HBM traffic per chain-iteration: y twice (16n) + x once (8n) +
// thread prefixes (6.2n) against the algorithmic 32n of SURVEY §8d.  DESIGN.md gives the op and byte accounting.
#include "../../include/omc.h"
#include "omc_common.cuh"
#include "omc_internal.h"
#include "omc_logtab.cuh"

namespace {

constexpr int TG_K = 18;                   // consecutive elements per thread (K/2 odd: 16-byte LDS stay conflict-free)
constexpr int TG_NT = 128;                 // threads per CTA, in all three kernels
constexpr int TG_NW = TG_NT / 32;
constexpr int TG_TILE = TG_K * TG_NT;      // 2304 elements = 18432 bytes per staged array
constexpr int TG_PAIRS = TG_K / 2;
constexpr unsigned FULL = 0xffffffffu;
constexpr int TG_AGG_G = 2;                // chains per CTA of the aggregate kernel (the shared P tile is staged once)
constexpr int TG_AGG_NORM = 4;             // thread aggregate: power-of-two renormalisation after element pair 4 (and at the
                                           // end); entries grow like u^k, so one mid-way stop keeps |d| up to 1e30 in range
constexpr int TG_LB_WIN = 4;               // successors polled in the first look-back round
constexpr int TG_SOLVE_MINB = 4;           // resident solve CTAs per SM the register allocation aims at (lean variant)

// Look-back record of one tile.  Every payload travels in ONE 16-byte word together with its flag (16-byte accesses
// are single transactions), so neither the writer nor the readers need a fence:
//   flag = epoch*4 + 1 on (a, b): affine aggregate ready, x_first = a * x_in + b  (x_in = first x of the next tile)
//   flag = epoch*4 + 2 on x     : x_first itself ready
struct __align__(64) RecB {
  double a; unsigned long long fa;
  double b; unsigned long long fb;
  double x; unsigned long long fx;
  double pad[2];
};

struct Workspace {
  unsigned long long epoch;   // advanced by the tile-scan kernel of every draw
  unsigned int pad[14];
  // followed by: RecB[n_tiles][n_chains], per-tile partial sums double[n_tiles][n_chains][4],
  //              tile totals double[n_tiles][n_chains][8], tile inputs double2[n_tiles][n_chains],
  //              thread prefixes double[n_chains][n_tiles][7][TG_NT]
};

__host__ __device__ inline long long align_up(long long x, long long a) { return (x + a - 1) / a * a; }

struct Layout {
  long long off_recb, off_flags_end, off_parts, off_tt, off_sin, off_ex, total;
  long long n_tiles;    // tiles of TG_TILE elements per chain
};
__host__ __device__ inline Layout make_layout(int n_chains, long long n) {
  Layout L;
  L.n_tiles = (n + TG_TILE - 1) / TG_TILE;
  const long long tc = L.n_tiles * n_chains;
  L.off_recb = align_up(sizeof(Workspace), 128);
  L.off_flags_end = L.off_recb + tc * (long long)sizeof(RecB);
  L.off_parts = align_up(L.off_flags_end, 128);
  L.off_tt = align_up(L.off_parts + tc * 32, 128);
  L.off_sin = L.off_tt + tc * 64;
  L.off_ex = align_up(L.off_sin + tc * 16, 128);
  L.total = L.off_ex + tc * 7 * TG_NT * 8;
  return L;
}

// ---------------------------------------------------------------------------------------------- small operators
// Transfer matrix of the projective recurrence on (p, q, h):  p' = a p + b q,  q' = c p + d q,  h' = e p + f q + g h.
struct TM { double a, b, c, d, e, f, g; };
struct Aff { double a, b; };  // v -> a v + b

__device__ __forceinline__ TM tm_identity() { return TM{1.0, 0.0, 0.0, 1.0, 0.0, 0.0, 1.0}; }
// left-multiply by the map of one element: p' = dd p - e2 q, q' = p, h' = bb p - ee h
__device__ __forceinline__ void tm_step(TM& t, double dd, double e2, double bb, double ee) {
  const double na = fma(dd, t.a, -(e2 * t.c));
  const double nb = fma(dd, t.b, -(e2 * t.d));
  const double ne = fma(bb, t.a, -(ee * t.e));
  const double nf = fma(bb, t.b, -(ee * t.f));
  t.c = t.a; t.d = t.b; t.a = na; t.b = nb; t.e = ne; t.f = nf; t.g = -(ee * t.g);
}
__device__ __forceinline__ TM tm_mul(const TM& x, const TM& y) {  // x after y
  TM r;
  r.a = fma(x.a, y.a, x.b * y.c);
  r.b = fma(x.a, y.b, x.b * y.d);
  r.c = fma(x.c, y.a, x.d * y.c);
  r.d = fma(x.c, y.b, x.d * y.d);
  r.e = fma(x.e, y.a, fma(x.f, y.c, x.g * y.e));
  r.f = fma(x.e, y.b, fma(x.f, y.d, x.g * y.f));
  r.g = x.g * y.g;
  return r;
}
// scale by a power of two so that the projective block (a b c d) has magnitude ~1 (exact; entries grow like u^k)
__device__ __forceinline__ void tm_normalize(TM& t) {
  // the high words of |a| .. |d| order like the magnitudes: the largest exponent comes out of three integer max
  const int hmx = max(max(__double2hiint(t.a) & 0x7fffffff, __double2hiint(t.b) & 0x7fffffff),
                      max(__double2hiint(t.c) & 0x7fffffff, __double2hiint(t.d) & 0x7fffffff));
  int ex = (hmx >> 20) - 1023;
  ex = max(-1000, min(1000, ex));
  const double s = __hiloint2double((1023 - ex) << 20, 0);
  t.a *= s; t.b *= s; t.c *= s; t.d *= s; t.e *= s; t.f *= s; t.g *= s;
}
__device__ __forceinline__ Aff aff_mul(const Aff& x, const Aff& y) { return Aff{x.a * y.a, fma(x.a, y.b, x.b)}; }  // x after y

__device__ __forceinline__ double shfl_d(double v, int src) { return __shfl_sync(FULL, v, src); }
__device__ __forceinline__ double shfl_up_d(double v, int d) { return __shfl_up_sync(FULL, v, d); }
__device__ __forceinline__ double shfl_dn_d(double v, int d) { return __shfl_down_sync(FULL, v, d); }
__device__ __forceinline__ TM tm_shfl(const TM& t, int src) {
  return TM{shfl_d(t.a, src), shfl_d(t.b, src), shfl_d(t.c, src), shfl_d(t.d, src), shfl_d(t.e, src), shfl_d(t.f, src),
            shfl_d(t.g, src)};
}
__device__ __forceinline__ TM tm_shfl_up(const TM& t, int d) {
  return TM{shfl_up_d(t.a, d), shfl_up_d(t.b, d), shfl_up_d(t.c, d), shfl_up_d(t.d, d), shfl_up_d(t.e, d),
            shfl_up_d(t.f, d), shfl_up_d(t.g, d)};
}

// 16-byte (payload, flag) words of the look-back records: one transaction each way, no fences
__device__ __forceinline__ void st_word(void* p, double v, unsigned long long flag) {
  asm volatile("st.relaxed.gpu.global.v2.u64 [%0], {%1, %2};" ::"l"(p), "l"(__double_as_longlong(v)), "l"(flag) : "memory");
}
__device__ __forceinline__ void ld_word(const void* p, double& v, unsigned long long& flag) {
  long long bits;
  asm volatile("ld.relaxed.gpu.global.v2.u64 {%0, %1}, [%2];" : "=l"(bits), "=l"(flag) : "l"(p) : "memory");
  v = __longlong_as_double(bits);
}
// issue-now read-only load: volatile asm keeps it where it is written (ahead of the RNG work that hides its latency)
__device__ __forceinline__ double ld_nc_now(const double* p) {
  double v;
  asm volatile("ld.global.nc.f64 %0, [%1];" : "=d"(v) : "l"(p));
  return v;
}

// 1/sqrt(u): MUFU.RSQ64H seed (~2^-22) + one third-order step (relative error ~1e-16; not correctly rounded, which the
// 1e-10 parity bar does not need).  u <= 0 or NaN gives NaN/inf and is reported through the status word.
__device__ __forceinline__ double fast_rsqrt(double u) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(u));
  // one third-order step: with eps = 1 - u y^2 (|eps| ~ 2^-22), u^-1/2 = y (1 + eps/2 + 3 eps^2/8) + O(eps^3)
  const double eps = fma(-u, y * y, 1.0);
  y = fma(y, eps * fma(0.375, eps, 0.5), y);
  return y;
}

// ---- mbarrier + bulk async copies (TMA engine, SASS UBLKCP)
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "TG_WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra TG_WAIT_DONE;\n"
      "bra TG_WAIT_LOOP;\n"
      "TG_WAIT_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void bulk_s2g(void* gdst, const void* smem_src, unsigned bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n" ::"l"(gdst), "r"(smem_u32(smem_src)),
               "r"(bytes)
               : "memory");
  asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
}
__device__ __forceinline__ void bulk_store_wait() { asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory"); }
__device__ __forceinline__ bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// ---------------------------------------------------------------------------------------------- tile staging
// Shared-memory map (doubles): [0] mbarrier, [2..3] slot in front of pe (pe[-1]), then TG_TILE doubles per array.
struct Stage {
  const double* src;   // element 0 of this chain's array (nullptr => constant fill)
  long long limit;     // number of valid elements in the array
  double fill;
  double* dst;
};

// Stage CNT arrays for the tile starting at element i_t.  Full interior tiles with 16-byte aligned sources go through
// cp.async.bulk (issued here, completion on `bar`); everything else (last tile, odd alignments, absent arrays) through
// plain loads.  Returns whether the bulk path was taken; stage_wait() makes the data visible to every thread.
template <int CNT>
__device__ __forceinline__ bool stage_issue(const Stage (&st)[CNT], long long i_t, long long n, unsigned long long* bar,
                                            int tid, int n_threads) {
  bool bulk = (i_t + TG_TILE < n);
#pragma unroll
  for (int q = 0; q < CNT; ++q)
    if (st[q].dst && st[q].src) bulk = bulk && al16(st[q].src + i_t) && (i_t + TG_TILE <= st[q].limit);
  if (bulk) {
    if (tid == 0) {
      unsigned bytes = 0;
#pragma unroll
      for (int q = 0; q < CNT; ++q)
        if (st[q].dst && st[q].src) bytes += TG_TILE * 8;
      mbar_expect_tx(bar, bytes);
#pragma unroll
      for (int q = 0; q < CNT; ++q)
        if (st[q].dst && st[q].src) bulk_g2s(st[q].dst, st[q].src + i_t, TG_TILE * 8, bar);
    }
  }
#pragma unroll
  for (int q = 0; q < CNT; ++q) {
    if (!st[q].dst || (st[q].src && bulk)) continue;
    for (int j = tid; j < TG_TILE; j += n_threads) {
      const long long i = i_t + j;
      st[q].dst[j] = (st[q].src && i < st[q].limit) ? __ldg(st[q].src + i) : st[q].fill;
    }
  }
  return bulk;
}
__device__ __forceinline__ void stage_wait(bool bulk, unsigned long long* bar) {
  if (bulk) mbar_wait(bar, 0);
  __syncthreads();
}

// ---------------------------------------------------------------------------------------------- normals
// Counter of Philox block `block` of a chain: position based (the draw does not depend on tiling or sharding); blocks
// beyond 2^20 spill into the second counter word.
__device__ __forceinline__ uint4 normal_counter(unsigned long long sw, unsigned int gchain, unsigned int site,
                                                unsigned long long block) {
  return make_uint4((unsigned int)sw, (unsigned int)(sw >> 32) ^ (unsigned int)(block >> 20) * 0x9E3779B9u, gchain,
                    (site << 20) | (unsigned int)(block & 0xFFFFFu));
}
__device__ __forceinline__ uint4 normal_block(unsigned long long sw, uint2 key, unsigned int gchain, unsigned int site,
                                              unsigned long long block) {
  return philox4x32_10(normal_counter(sw, gchain, site, block), key);
}
// Philox4x32-10 on G counter blocks in lock-step: G independent multiply chains in flight per thread (one block at a
// time leaves the thread waiting on every dependent IMAD.WIDE -> LOP3 pair).  Same values as philox4x32_10.
template <int G>
__device__ __forceinline__ void philox_group(uint4 (&ctr)[G], uint2 key) {
  const unsigned int M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
#pragma unroll
    for (int i = 0; i < G; ++i) {
      const unsigned int hi0 = __umulhi(M0, ctr[i].x), lo0 = M0 * ctr[i].x;
      const unsigned int hi1 = __umulhi(M1, ctr[i].z), lo1 = M1 * ctr[i].z;
      ctr[i] = make_uint4(hi1 ^ ctr[i].y ^ key.x, lo1, hi0 ^ ctr[i].w ^ key.y, lo0);
    }
    key.x += W0;
    key.y += W1;
  }
}
// Two normals by Box-Muller in fp64 with purpose-built pieces (tools/rng_model.py is the numpy model), from
// U = mm 2^-jp1 (mm in [1, 2), idx = its top 7 mantissa bits) and the angle bits in b.w, b.z:
//   -ln U   : ln m = lc[i] + ln1p(m rc[i] - 1) with a 128-entry table on the top 7 mantissa bits and a degree-7 series
//             (|m rc - 1| <= 2^-8); absolute error 2e-15
//   radius  : sqrt(2E) = 2E * rsqrt(2E)
//   angle   : uniform in the first octant from 52 bits (Taylor sin / cos to 1 ulp on [0, pi/4]), three more bits swap
//             sin <-> cos and pick the two signs
__device__ __forceinline__ void normal_from(double jp1, double mm, int idx, uint4 b, double& z0, double& z1) {
  // ---- radius
  const double2 tab = __ldg(reinterpret_cast<const double2*>(omc_logtab) + idx);
  const double rr = fma(mm, tab.x, -1.0);
  double p = fma(rr, 1.0 / 7.0, -1.0 / 6.0);
  p = fma(p, rr, 1.0 / 5.0);
  p = fma(p, rr, -1.0 / 4.0);
  p = fma(p, rr, 1.0 / 3.0);
  p = fma(p, rr, -1.0 / 2.0);
  p = fma(p, rr, 1.0);
  const double lnm = fma(p, rr, tab.y);
  const double en = fma(jp1, 0.6931471805599453094, -lnm);     // E = -ln U  (>= -2e-15)
  const double e2 = fma(2.0, en, 0x1p-47);                     // 2E, kept strictly positive
  const double rad = e2 * fast_rsqrt(e2);
  // ---- angle: 52 bits = low 20 of w : z
  const double fr = __hiloint2double((int)((b.w & 0x000FFFFFu) | 0x3FF00000u), (int)b.z) - 1.0;
  const double phi = fr * 0.78539816339744830962;
  const double x2 = phi * phi;
  double ps = fma(x2, -1.0 / 1307674368000.0, 1.0 / 6227020800.0);
  ps = fma(ps, x2, -1.0 / 39916800.0);
  ps = fma(ps, x2, 1.0 / 362880.0);
  ps = fma(ps, x2, -1.0 / 5040.0);
  ps = fma(ps, x2, 1.0 / 120.0);
  ps = fma(ps, x2, -1.0 / 6.0);
  ps = fma(ps, x2, 1.0);
  double pc = fma(x2, 1.0 / 20922789888000.0, -1.0 / 87178291200.0);
  pc = fma(pc, x2, 1.0 / 479001600.0);
  pc = fma(pc, x2, -1.0 / 3628800.0);
  pc = fma(pc, x2, 1.0 / 40320.0);
  pc = fma(pc, x2, -1.0 / 720.0);
  pc = fma(pc, x2, 1.0 / 24.0);
  pc = fma(pc, x2, -0.5);
  pc = fma(pc, x2, 1.0);
  ps *= phi;
  const bool swp = (b.w >> 20) & 1u;
  const double cs = swp ? ps : pc, sn = swp ? pc : ps;
  const double a0 = rad * cs, a1 = rad * sn;
  z0 = __hiloint2double(__double2hiint(a0) ^ (int)((b.w << 10) & 0x80000000u), __double2loint(a0));
  z1 = __hiloint2double(__double2hiint(a1) ^ (int)((b.w << 9) & 0x80000000u), __double2loint(a1));
}

// ---------------------------------------------------------------------------------------------- fp32-assisted normals
// Generator of the solve kernel: FOUR normals per Philox4x32-10 block, Box-Muller with the transcendental parts on the
// special-function unit in fp32 (lg2 / sqrt / sin / cos.approx, absolute error ~2^-21 each), the product r * (cos, sin)
// formed in fp64 from the exactly converted factors.  The distribution differs from N(0,1) by ~1e-7 in Kolmogorov
// distance (what curand_normal gives), invisible to any run shorter than ~1e13 draws per element, in exchange for ~45
// of the 68 instructions per element of all-fp64 pairs.  Both generators it was measured against were removed:
// all-fp64 Box-Muller pairs (normal_from for every pair) took 0.607 ms per C3 draw against 0.522 ms
// (profiles/r02_tridiag_variants.txt); a Marsaglia-Tsang ziggurat had already lost to those pairs, 0.69 ms (256
// layers) and 0.76 ms (1024 layers) against 0.605 ms at 64 x 1e6 -- the FP64-pipe share of the kernel fell from 46 % to
// 23 %, but its random 16-byte table gathers doubled the long-scoreboard stalls and the instruction count did not fall
// (profiles/r02_tridiag_ziggurat_variants.txt).  Stream layout: the thread's TG_K consecutive elements (a
// "group") take blocks group * TG_F32_BLOCKS + k; words (x, y) of a block make elements 4k, 4k+1 of the group and
// (z, w) elements 4k+2, 4k+3 -- a fixed function of the element index, independent of tiling and sharding.
// A pair whose radius word is below 2^12 (probability 2^-20) is redone in fp64 with 32 more bits below it, so the
// tail of the radius is exact beyond 6 sigma as well.
constexpr int TG_F32_BLOCKS = (TG_PAIRS + 1) / 2;
constexpr int TG_F32_GROUP = 3;            // Philox blocks advanced in lock-step per thread
__device__ __forceinline__ bool normal_pair_f32(unsigned int w1, unsigned int w2, double& z0, double& z1) {
  const unsigned int fb = __float_as_uint(__uint2float_rz(w1));                       // top 24 bits of w1, exactly
  const float mant = __uint_as_float((fb & 0x007FFFFFu) | 0x3F800000u);               // [1, 2)
  const float jp1 = __uint_as_float(0x4B000000u | (159u - (fb >> 23))) - 8388608.0f;  // 1 + leading zeros of w1
  float lg, r, sn, cs;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(mant));
  const float e2 = (jp1 - lg) * 1.38629436111989f;                                    // -2 ln U, U = mant 2^-(j+1)
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e2));
  const float th = (float)(int)w2 * 1.4629180792671596e-9f;                           // [-pi, pi]: 2 pi 2^-32
  asm("sin.approx.ftz.f32 %0, %1;" : "=f"(sn) : "f"(th));
  asm("cos.approx.ftz.f32 %0, %1;" : "=f"(cs) : "f"(th));
  const double rd = (double)r;
  z0 = rd * (double)cs;
  z1 = rd * (double)sn;
  return w1 >= (1u << 12);
}
__device__ __noinline__ double2 normal_pair_f32_slow(unsigned long long sw, uint2 key, unsigned int gchain,
                                                     unsigned int site, unsigned long long block, int half) {
  const uint4 b = normal_block(sw, key, gchain, site, block);
  const uint4 b2 = normal_block(sw, make_uint2(key.x ^ 0x5A1C0DE5u, key.y + 1u), gchain, site, block);
  const unsigned int w1 = half ? b.z : b.x, w2 = half ? b.w : b.y;
  const unsigned long long r = ((unsigned long long)w1 << 32) | (half ? b2.z : b2.x);
  const int j = __clzll((long long)r);
  const unsigned long long sh = (j >= 63) ? 0ull : (r << (j + 1));
  const unsigned long long mb = sh >> 12;
  const double mm = __longlong_as_double((long long)(0x3FF0000000000000ull | mb));
  double2 z;
  normal_from((double)(j + 1), mm, (int)(mb >> 45), make_uint4(0u, 0u, half ? b2.w : b2.y, w2), z.x, z.y);
  return z;
}

// ---------------------------------------------------------------------------------------------- tile scan
// Exclusive scan of one chain's tile totals -> (u, f) entering every tile, by the NT threads of one CTA (a kernel of
// its own, one CTA per chain: 11 us between the two big kernels.  Folding it into the aggregate kernel's tail -- the
// CTA that finishes a chain's last tile scans it, fence + atomic hand-over -- MEASURED slower, 0.240 against 0.177 ms
// for aggregate + scan: with tile-major work every chain finishes in the last wave, so nothing is hidden, and the
// fence sits in every CTA; profiles/r02_tridiag_variants.txt).
template <int NT>
__device__ __forceinline__ void tilescan_chain(Workspace* ws, const Layout& L, int C, int chain, int tid,
                                               double (&s_tot)[NT / 32][7]) {
  const int lane = tid & 31, warp = tid >> 5;
  if (chain == 0 && tid == 0) ws->epoch = ws->epoch + 1;   // fresh flag values for the solve kernel that follows
  char* wsb = reinterpret_cast<char*>(ws);
  const double* tt = reinterpret_cast<const double*>(wsb + L.off_tt);
  double2* sin_ = reinterpret_cast<double2*>(wsb + L.off_sin);
  const long long T = L.n_tiles;
  const long long per = (T + NT - 1) / NT;
  TM agg = tm_identity();
  for (long long q = 0; q < per; ++q) {
    const long long t = tid * per + q;
    if (t < T) {
      const double* p = tt + (t * C + chain) * 8;
      agg = tm_mul(TM{__ldcg(p), __ldcg(p + 1), __ldcg(p + 2), __ldcg(p + 3), __ldcg(p + 4), __ldcg(p + 5), __ldcg(p + 6)}, agg);
      tm_normalize(agg);
    }
  }
  TM inc = agg;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const TM o = tm_shfl_up(inc, d);
    if (lane >= d) {
      inc = tm_mul(inc, o);
      tm_normalize(inc);
    }
  }
  if (lane == 31) {
    s_tot[warp][0] = inc.a; s_tot[warp][1] = inc.b; s_tot[warp][2] = inc.c; s_tot[warp][3] = inc.d;
    s_tot[warp][4] = inc.e; s_tot[warp][5] = inc.f; s_tot[warp][6] = inc.g;
  }
  __syncthreads();
  TM wex = tm_identity();
  for (int w = 0; w < warp; ++w) {
    const TM ww{s_tot[w][0], s_tot[w][1], s_tot[w][2], s_tot[w][3], s_tot[w][4], s_tot[w][5], s_tot[w][6]};
    wex = tm_mul(ww, wex);
    tm_normalize(wex);
  }
  TM ex = tm_shfl_up(inc, 1);
  if (lane == 0) ex = tm_identity();
  ex = tm_mul(ex, wex);
  // state entering the thread's first tile, from the initial state (u, q, f) = (1, 1, 0)
  double u, f;
  {
    const double p0 = ex.a + ex.b, q0 = ex.c + ex.d, h0 = ex.e + ex.f;
    u = p0 / q0;
    f = h0 / q0;
  }
  for (long long q = 0; q < per; ++q) {
    const long long t = tid * per + q;
    if (t < T) {
      sin_[t * C + chain] = make_double2(u, f);
      const double* p = tt + (t * C + chain) * 8;
      const double pp = fma(__ldcg(p), u, __ldcg(p + 1)), qq = fma(__ldcg(p + 2), u, __ldcg(p + 3)),
                   hh = fma(__ldcg(p + 4), u, fma(__ldcg(p + 6), f, __ldcg(p + 5)));
      u = pp / qq;
      f = hh / qq;
    }
  }
}

constexpr int TS_NT = 256;
__global__ void __launch_bounds__(TS_NT) tg_tilescan_kernel(Workspace* ws, Layout L, int C) {
  __shared__ double s_tot[TS_NT / 32][7];
  tilescan_chain<TS_NT>(ws, L, C, (int)blockIdx.x, (int)threadIdx.x, s_tot);
}

// ---------------------------------------------------------------------------------------------- aggregate kernel
// The compute part of the aggregate kernel: thread aggregate over 18 staged elements, CTA scan, stores.  (A separate
// function: written inline in the kernel, the same code allocates registers differently.)
template <bool GENERAL, int G>
__device__ __forceinline__ void aggregate_compute(const omc_tridiag_nn_t& a, char* wsb, const Layout& L,
                                                  double (&s_tot)[G][TG_NW][7], const double* spe, const double* spd,
                                                  const double* sy, const double* sw, const double* sh, double lam,
                                                  double tau, int sub, int tid, bool live, int chain, long long tile) {
  const int lane = tid & 31, warp = tid >> 5;
  const int C = a.n_chains;
  // ---- thread aggregate over its 18 elements (no divisions)
  const int j0 = tid * TG_K;
  TM t = tm_identity();
  {
    double eprev = lam * spe[j0 - 1];
#pragma unroll
    for (int c = 0; c < TG_PAIRS; ++c) {
      const double2 pd2 = *reinterpret_cast<const double2*>(spd + j0 + 2 * c);
      const double2 pe2 = *reinterpret_cast<const double2*>(spe + j0 + 2 * c);
      const double2 y2 = *reinterpret_cast<const double2*>(sy + j0 + 2 * c);
      double2 w2 = make_double2(1.0, 1.0), h2 = make_double2(0.0, 0.0);
      if (GENERAL) {
        w2 = *reinterpret_cast<const double2*>(sw + j0 + 2 * c);
        h2 = *reinterpret_cast<const double2*>(sh + j0 + 2 * c);
      }
      {
        const double tw = GENERAL ? tau * w2.x : tau;
        const double dd = fma(lam, pd2.x, tw);
        const double bb = GENERAL ? fma(lam, h2.x, tw * y2.x) : tw * y2.x;
        tm_step(t, dd, eprev * eprev, bb, eprev);
        eprev = lam * pe2.x;
      }
      {
        const double tw = GENERAL ? tau * w2.y : tau;
        const double dd = fma(lam, pd2.y, tw);
        const double bb = GENERAL ? fma(lam, h2.y, tw * y2.y) : tw * y2.y;
        tm_step(t, dd, eprev * eprev, bb, eprev);
        eprev = lam * pe2.y;
      }
      if (c == TG_AGG_NORM) tm_normalize(t);
    }
    tm_normalize(t);
  }
  // ---- CTA scan of the transfer matrices (thread order): inclusive within the warp, then across the 4 warps.
  //      Normalised inputs grow by < 2^63 over the five levels of the warp scan, so it renormalises only at the end.
  TM inc = t;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const TM o = tm_shfl_up(inc, d);
    if (lane >= d) inc = tm_mul(inc, o);
  }
  tm_normalize(inc);
  if (lane == 31) {
    s_tot[sub][warp][0] = inc.a; s_tot[sub][warp][1] = inc.b; s_tot[sub][warp][2] = inc.c; s_tot[sub][warp][3] = inc.d;
    s_tot[sub][warp][4] = inc.e; s_tot[sub][warp][5] = inc.f; s_tot[sub][warp][6] = inc.g;
  }
  __syncthreads();
  TM wex = tm_identity();   // composition of the warps below this one
  for (int w = 0; w < warp; ++w) {
    const TM ww{s_tot[sub][w][0], s_tot[sub][w][1], s_tot[sub][w][2], s_tot[sub][w][3], s_tot[sub][w][4], s_tot[sub][w][5], s_tot[sub][w][6]};
    wex = tm_mul(ww, wex);
  }
  TM ex = tm_shfl_up(inc, 1);
  if (lane == 0) ex = tm_identity();
  ex = tm_mul(ex, wex);       // exclusive prefix of this thread inside the tile
  tm_normalize(ex);
  if (live) {
    double* exg = reinterpret_cast<double*>(wsb + L.off_ex) + ((long long)chain * L.n_tiles + tile) * 7 * TG_NT + tid;
    exg[0 * TG_NT] = ex.a; exg[1 * TG_NT] = ex.b; exg[2 * TG_NT] = ex.c; exg[3 * TG_NT] = ex.d;
    exg[4 * TG_NT] = ex.e; exg[5 * TG_NT] = ex.f; exg[6 * TG_NT] = ex.g;
  }
  if (live && tid == TG_NT - 1) {     // tile total = the last thread's inclusive prefix
    TM tot = tm_mul(inc, wex);
    tm_normalize(tot);
    double* tt = reinterpret_cast<double*>(wsb + L.off_tt) + (tile * C + chain) * 8;
    tt[0] = tot.a; tt[1] = tot.b; tt[2] = tot.c; tt[3] = tot.d; tt[4] = tot.e; tt[5] = tot.f; tt[6] = tot.g;
  }
}

// G chains per CTA (G x TG_NT threads): the tile of the shared P is staged ONCE for the G chains, which halves (G = 2)
// or quarters (G = 4) the shared memory per resident warp -- this kernel is a load -> compute -> store pipeline whose
// only latency hiding is the number of CTAs resident next to each other.  GENERAL (weights / prior mean) keeps G = 1.
template <bool GENERAL, int G>
__global__ void __launch_bounds__(TG_NT* G) tg_aggregate_kernel(omc_tridiag_nn_t a, Workspace* ws, Layout L, int n_groups) {
  static_assert(!GENERAL || G == 1, "GENERAL aggregate kernel stages per-chain arrays for one chain only");
  extern __shared__ __align__(128) double sm[];
  __shared__ double s_tot[G][TG_NW][7];
  unsigned long long* bar = reinterpret_cast<unsigned long long*>(sm);
  double* spe = sm + 4;
  double* spd = spe + TG_TILE;
  double* sy0 = spd + TG_TILE;     // G tiles of y, one per chain of the group
  double* sw = sy0 + TG_TILE;      // GENERAL only
  double* sh = sw + TG_TILE;       // GENERAL only
  const int sub = threadIdx.x / TG_NT;            // which chain of the group
  const int tid = threadIdx.x % TG_NT;
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  __syncthreads();
  const int C = a.n_chains;
  const long long tile = blockIdx.x / n_groups;   // tile-major: the chains read the same tile of the shared P together
  const int chain0 = (int)(blockIdx.x % n_groups) * G;
  const int chain = chain0 + sub;
  const bool live = chain < C;                    // ragged last group
  const int cc = live ? chain : C - 1;
  const long long n = a.n;
  char* wsb = reinterpret_cast<char*>(ws);
  const long long i_t = tile * TG_TILE;
  const double lam = a.lambda.ptr ? a.lambda.ptr[(long long)cc * a.lambda.chain_stride] : 1.0;
  const double tau = a.tau.ptr ? a.tau.ptr[(long long)cc * a.tau.chain_stride] : 1.0;
  double* sy = sy0 + sub * TG_TILE;

  if (threadIdx.x == 0) spe[-1] = (a.pe && i_t > 0 && i_t - 1 < n - 1) ? __ldg(a.pe + i_t - 1) : 0.0;
  bool bulk;
  if (GENERAL) {
    const double* yp = a.y.ptr + (long long)cc * a.y.chain_stride;
    const Stage st[5] = {{a.pe, n - 1, 0.0, spe}, {a.pd, n, 1.0, spd}, {yp, n, 0.0, sy},
                         {a.w.ptr ? a.w.ptr + (long long)cc * a.w.chain_stride : nullptr, n, 1.0, sw},
                         {a.h.ptr ? a.h.ptr + (long long)cc * a.h.chain_stride : nullptr, n, 0.0, sh}};
    bulk = stage_issue<5>(st, i_t, n, bar, threadIdx.x, TG_NT * G);
  } else {
    Stage st[2 + G];
    st[0] = Stage{a.pe, n - 1, 0.0, spe};
    st[1] = Stage{a.pd, n, 1.0, spd};
#pragma unroll
    for (int g = 0; g < G; ++g)
      st[2 + g] = Stage{a.y.ptr + (long long)min(chain0 + g, C - 1) * a.y.chain_stride, n, 0.0, sy0 + g * TG_TILE};
    bulk = stage_issue<2 + G>(st, i_t, n, bar, threadIdx.x, TG_NT * G);
  }
  stage_wait(bulk, bar);

  aggregate_compute<GENERAL, G>(a, wsb, L, s_tot, spe, spd, sy, sw, sh, lam, tau, sub, tid, live, chain, tile);
}

// ---------------------------------------------------------------------------------------------- solve kernel
// GENERAL: diagonal weights w, prior-mean terms h = P mu0 and mu0 are staged too (absent ones are filled with 1 / 0).
// DEBUG  : injected normals (debug_z), log-det / factor probes, and the factorisation-only mode (x == NULL).
// Tiles are taken in blockIdx order, top tile first: the reverse look-back of a tile waits only on tiles with a LOWER
// block index, which the hardware dispatches earlier (the usual assumption of single-pass scans).
template <bool GENERAL, bool DEBUG>
__global__ void __launch_bounds__(TG_NT, DEBUG ? 1 : (GENERAL ? 2 : TG_SOLVE_MINB))
tg_solve_kernel(omc_tridiag_nn_t a, Workspace* ws, Layout L) {
  extern __shared__ __align__(128) double sm[];
  __shared__ double s_red[2 * TG_NW];
  __shared__ double s_part[3 * TG_NW];
  __shared__ int s_bad;
  unsigned long long* bar = reinterpret_cast<unsigned long long*>(sm);
  double* spe = sm + 4;
  double* spd = spe + TG_TILE;
  double* sy = spd + TG_TILE;
  double* sz = sy + TG_TILE;                          // DEBUG: the injected debug_z tile
  double* sw = DEBUG ? sz + TG_TILE : sz;             // GENERAL
  double* sh = sw + TG_TILE;                          // GENERAL
  double* smu = sh + TG_TILE;                         // GENERAL (TG_TILE + 2: mu0 of the next tile's first element)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned long long epoch = *reinterpret_cast<volatile unsigned long long*>(&ws->epoch);
  const int C = a.n_chains;
  const long long T = L.n_tiles;             // tiles per chain
  const long long work = blockIdx.x;
  const long long tile = T - 1 - work / C;   // top tiles first; tile-major over the chains
  const int chain = (int)(work % C);
  const long long n = a.n;
  char* wsb = reinterpret_cast<char*>(ws);
  RecB* recs = reinterpret_cast<RecB*>(wsb + L.off_recb);
  RecB* rec = recs + tile * C + chain;
  double* parts = reinterpret_cast<double*>(wsb + L.off_parts) + (tile * C + chain) * 4;
  const unsigned long long FLAG_A = epoch * 4 + 1, FLAG_P = epoch * 4 + 2;
  const long long i_t = tile * TG_TILE;
  const bool solve = !DEBUG || a.x != nullptr;
  const bool inject = DEBUG && a.debug_z != nullptr;
  const int j0 = tid * TG_K;
  const long long i0 = i_t + j0;
  const int nvalid = (int)max(0ll, min((long long)TG_K, n - i0));   // this thread's elements inside the chain

  // ---- stage the tile (thread 0 issues the bulk copies; nobody waits yet)
  bool bulk;
  {
    const double* yp = a.y.ptr + (long long)chain * a.y.chain_stride;
    const double* wp = (GENERAL && a.w.ptr) ? a.w.ptr + (long long)chain * a.w.chain_stride : nullptr;
    const double* hp = (GENERAL && a.h.ptr) ? a.h.ptr + (long long)chain * a.h.chain_stride : nullptr;
    const double* mp = (GENERAL && a.mu0.ptr) ? a.mu0.ptr + (long long)chain * a.mu0.chain_stride : nullptr;
    const double* zp = nullptr;
    if (inject) {
      const long long sw_ = a.rng.sweep ? (long long)(*a.rng.sweep) : 0ll;
      zp = a.debug_z + sw_ * a.debug_sweep_stride + (long long)chain * n;
    }
    if (tid == 0) {
      s_bad = 0;
      mbar_init(bar, 1);
      asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
      spe[-1] = (a.pe && i_t > 0 && i_t - 1 < n - 1) ? __ldg(a.pe + i_t - 1) : 0.0;
      if (GENERAL) smu[TG_TILE] = (mp && i_t + TG_TILE < n) ? __ldg(mp + i_t + TG_TILE) : 0.0;
    }
    const Stage st[7] = {{a.pe, n - 1, 0.0, spe},
                         {a.pd, n, 1.0, spd},
                         {yp, n, 0.0, sy},
                         {wp, n, 1.0, GENERAL ? sw : nullptr},
                         {hp, n, 0.0, GENERAL ? sh : nullptr},
                         {mp, n, 0.0, GENERAL ? smu : nullptr},
                         {zp, n, 0.0, inject ? sz : nullptr}};
    bulk = stage_issue<7>(st, i_t, n, bar, tid, TG_NT);
  }
  // ---- loads of the thread prefix / tile input / scalars go out now; their latency hides under the normals
  const double* exg = reinterpret_cast<const double*>(wsb + L.off_ex) + ((long long)chain * L.n_tiles + tile) * 7 * TG_NT + tid;
  const double* sin_p = reinterpret_cast<const double*>(wsb + L.off_sin) + (tile * C + chain) * 2;
  const double ea = ld_nc_now(exg), eb = ld_nc_now(exg + TG_NT), ec = ld_nc_now(exg + 2 * TG_NT),
               ed = ld_nc_now(exg + 3 * TG_NT), ee = ld_nc_now(exg + 4 * TG_NT), ef = ld_nc_now(exg + 5 * TG_NT),
               eg = ld_nc_now(exg + 6 * TG_NT);
  const double sin_x = ld_nc_now(sin_p), sin_y = ld_nc_now(sin_p + 1);
  const double lam = a.lambda.ptr ? ld_nc_now(a.lambda.ptr + (long long)chain * a.lambda.chain_stride) : 1.0;
  const double tau = a.tau.ptr ? ld_nc_now(a.tau.ptr + (long long)chain * a.tau.chain_stride) : 1.0;
  // ---- this thread's 18 normals, drawn into registers while the tile loads are in flight
  double g[TG_K], m[TG_K];
  if (!inject && solve && nvalid > 0) {
    const unsigned long long sweep = a.rng.sweep ? *a.rng.sweep : 0ull;
    const uint2 key = make_uint2((unsigned int)a.rng.seed, (unsigned int)(a.rng.seed >> 32));
    const unsigned int gchain = a.rng.chain_offset + (unsigned int)chain;
    unsigned int redo = 0;
    const unsigned long long block0 = (unsigned long long)(i0 / TG_K) * TG_F32_BLOCKS;
#pragma unroll
    for (int k0 = 0; k0 < TG_F32_BLOCKS; k0 += TG_F32_GROUP) {
      uint4 b[TG_F32_GROUP];
#pragma unroll
      for (int i = 0; i < TG_F32_GROUP; ++i) b[i] = normal_counter(sweep, gchain, a.rng.site, block0 + k0 + i);
      philox_group<TG_F32_GROUP>(b, key);
#pragma unroll
      for (int i = 0; i < TG_F32_GROUP; ++i) {
        const int k = k0 + i;
        if (2 * k < TG_PAIRS && !normal_pair_f32(b[i].x, b[i].y, g[4 * k], g[4 * k + 1])) redo |= 1u << (2 * k);
        if (2 * k + 1 < TG_PAIRS && !normal_pair_f32(b[i].z, b[i].w, g[4 * k + 2], g[4 * k + 3])) redo |= 1u << (2 * k + 1);
      }
    }
    while (redo) {   // probability 2^-20 per pair
      const int c = __ffs(redo) - 1;
      redo &= redo - 1;
      const double2 z = normal_pair_f32_slow(sweep, key, gchain, a.rng.site, block0 + (c >> 1), c & 1);
#pragma unroll
      for (int cc = 0; cc < TG_PAIRS; ++cc)
        if (cc == c) { g[2 * cc] = z.x; g[2 * cc + 1] = z.y; }
    }
  } else {
#pragma unroll
    for (int k = 0; k < TG_K; ++k) g[k] = 0.0;
  }
  // ---- exact boundary values entering this thread's elements: 1/u_{i0-1} and f_{i0-1}
  double iu_prev, f_prev;
  {
    const double p = fma(ea, sin_x, eb), q = fma(ec, sin_x, ed), h = fma(ee, sin_x, fma(eg, sin_y, ef));
    iu_prev = q / p;
    f_prev = h / q;
  }
  __syncthreads();               // mbarrier initialised, plain-load fills visible
  if (bulk) mbar_wait(bar, 0);
  if (inject) {
#pragma unroll
    for (int c = 0; c < TG_PAIRS; ++c) {
      const double2 z2 = *reinterpret_cast<const double2*>(sz + j0 + 2 * c);
      g[2 * c] = z2.x;
      g[2 * c + 1] = z2.y;
    }
  }

  // ---- ascending pass over this thread's 18 elements.  The pivots run in scaled principal-minor form
  //        P_k = (s d_k) P_{k-1} - (s e_{k-1})^2 P_{k-2},   u_k = P_k / (s P_{k-1}),   s = 4^r ~ 1/u  (exact scaling)
  //      so that the only serial dependence is ONE fused multiply-add per element; 1/sqrt(u_k) = sqrt(s) P_{k-1} /
  //      sqrt(P_k P_{k-1}) and everything built on it (1/u, m, g) is independent work across the 18 elements.
  Aff bagg{1.0, 0.0};          // x_{i0} = bagg.a * x_{i0+18} + bagg.b
  bool bad = false;
  double logdet = 0.0;
  {
    int ex2 = (((__double2hiint(iu_prev) >> 20) & 0x7ff) - 1023) & ~1;
    ex2 = max(-600, min(600, ex2));
    const double s = __hiloint2double((1023 + ex2) << 20, 0);
    const double rs = __hiloint2double((1023 + ex2 / 2) << 20, 0);
    const double sl = s * lam, st = s * tau;
    double pm1 = 1.0, pm2 = iu_prev * __hiloint2double((1023 - ex2) << 20, 0);
    double eprev = lam * spe[j0 - 1];
    double mprev = eprev * iu_prev;
#pragma unroll
    for (int c = 0; c < TG_PAIRS; ++c) {
      const double2 pd2 = *reinterpret_cast<const double2*>(spd + j0 + 2 * c);
      const double2 pe2 = *reinterpret_cast<const double2*>(spe + j0 + 2 * c);
      const double2 y2 = *reinterpret_cast<const double2*>(sy + j0 + 2 * c);
      double2 w2 = make_double2(1.0, 1.0), h2 = make_double2(0.0, 0.0);
      if (GENERAL) {
        w2 = *reinterpret_cast<const double2*>(sw + j0 + 2 * c);
        h2 = *reinterpret_cast<const double2*>(sh + j0 + 2 * c);
      }
      if (c == 3 || c == 6) {   // keep the minors near 1 (exact power-of-two rescale)
        const int exp_ = max(-900, min(900, ((__double2hiint(pm1) >> 20) & 0x7ff) - 1023));
        const double sc = __hiloint2double((1023 - exp_) << 20, 0);
        pm1 *= sc;
        pm2 *= sc;
      }
#pragma unroll
      for (int hlf = 0; hlf < 2; ++hlf) {
        const int k = 2 * c + hlf;
        const double pdk = hlf ? pd2.y : pd2.x, pek = hlf ? pe2.y : pe2.x, yk = hlf ? y2.y : y2.x;
        const double wk = hlf ? w2.y : w2.x, hk = hlf ? h2.y : h2.x, zk = g[k];
        const double ds = GENERAL ? fma(sl, pdk, st * wk) : fma(sl, pdk, st);   // s d_k
        const double bb = GENERAL ? fma(lam, hk, tau * wk * yk) : tau * yk;
        const double es = s * eprev;                                            // s e_{k-1}
        const double pk = fma(ds, pm1, -((es * es) * pm2));
        const double tt = pk * pm1;
        if (!(tt > 0.0)) bad = true;       // pivot u_k <= 0 (or NaN)
        const double su = rs * (pm1 * fast_rsqrt(tt));
        const double iu = su * su;
        const double f = fma(-mprev, f_prev, bb);
        const double e = lam * pek;
        const double mk = e * iu;
        const double gk = fma(f, iu, zk * su);
        g[k] = gk;
        m[k] = mk;
        bagg.b = fma(bagg.a, gk, bagg.b);
        bagg.a = -(bagg.a * mk);
        if (DEBUG && k < nvalid) {
          const double u = 1.0 / iu;
          if (a.logdet) logdet += log(u);
          if (a.probe_l) a.probe_l[(long long)chain * n + i0 + k] = sqrt(u);
          if (a.probe_c && i0 + k < n - 1) a.probe_c[(long long)chain * (n - 1) + i0 + k] = e * su;
        }
        pm2 = pm1;
        pm1 = pk;
        f_prev = f;
        eprev = e;
        mprev = mk;
      }
    }
  }
  if (bad) s_bad = 1;

  double ssp = 0.0, ssp2 = 0.0, ssl = 0.0;
  bool bulk_out = false;
  if (solve) {
    // ---- CTA scan of the backward affine maps, from the top thread down; exclusive prefix = all HIGHER threads
    Aff inc = bagg;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const Aff o{shfl_dn_d(inc.a, d), shfl_dn_d(inc.b, d)};
      if (lane + d < 32) inc = aff_mul(inc, o);
    }
    if (lane == 0) { s_red[2 * warp] = inc.a; s_red[2 * warp + 1] = inc.b; }
    __syncthreads();
    Aff wex{1.0, 0.0};    // composition of the warps above this one
    Aff tot{1.0, 0.0};    // the whole tile
#pragma unroll
    for (int w = TG_NW - 1; w >= 0; --w) {
      if (w == warp) wex = tot;
      tot = aff_mul(Aff{s_red[2 * w], s_red[2 * w + 1]}, tot);
    }
    Aff lex{shfl_dn_d(inc.a, 1), shfl_dn_d(inc.b, 1)};
    if (lane == 31) lex = Aff{1.0, 0.0};
    const Aff bex = aff_mul(lex, wex);   // x_{i0+18} = bex.a * x_in + bex.b
    // ---- reverse look-back over the tiles of this chain, 32 successors per round.  Every warp walks it for itself
    //      (no CTA barrier, nobody idles); warp 0 publishes the tile's records.
    double xfar = 0.0;     // x beyond the last element is 0 (and its multiplier m_{n-1} is 0)
    Aff R{1.0, 0.0};
    if (tile < T - 1) {
      if (tid == 0) {
        st_word(&rec->a, tot.a, FLAG_A);
        st_word(&rec->b, tot.b, FLAG_A);
      }
      // The first round polls only the TG_LB_WIN nearest successors: the resolving record is almost always among them,
      // and records written long ago may have left L2 (a full-width first round paid a DRAM round trip for them).
      long long base = tile + 1;
      int win = TG_LB_WIN;
      while (true) {
        const long long j = base + lane;
        bool have_x = false;
        Aff mine{1.0, 0.0};
        double px = 0.0;
        if (lane < win) {
          have_x = true;                // beyond the chain's last tile: x = 0 terminates the walk
          if (j < T) {
            const RecB* pr = recs + j * C + chain;
            unsigned long long fa, fb, fx;
            while (true) {
              ld_word(&pr->x, px, fx);
              ld_word(&pr->a, mine.a, fa);
              ld_word(&pr->b, mine.b, fb);
              have_x = (fx == FLAG_P);
              if (have_x || (fa == FLAG_A && fb == FLAG_A)) break;
            }
          }
        }
        const unsigned pmask = __ballot_sync(FULL, have_x);
        const int lp = pmask ? (__ffs(pmask) - 1) : win;
        for (int l = 0; l < lp; ++l) R = aff_mul(R, Aff{shfl_d(mine.a, l), shfl_d(mine.b, l)});
        if (lp < win) {
          xfar = shfl_d(px, lp);
          break;
        }
        base += win;
        win = 32;
      }
    }
    const double x_in = fma(R.a, xfar, R.b);
    if (tid == 0) st_word(&rec->x, fma(tot.a, x_in, tot.b), FLAG_P);
    // ---- descending pass: x and both quadratic forms; x overwrites y in shared memory
    double xn = fma(bex.a, x_in, bex.b);
    double rn = GENERAL ? xn - smu[j0 + TG_K] : xn;
#pragma unroll
    for (int c = TG_PAIRS - 1; c >= 0; --c) {
      const double2 pd2 = *reinterpret_cast<const double2*>(spd + j0 + 2 * c);
      const double2 pe2 = *reinterpret_cast<const double2*>(spe + j0 + 2 * c);
      const double2 y2 = *reinterpret_cast<const double2*>(sy + j0 + 2 * c);
      double2 w2 = make_double2(1.0, 1.0), mu2 = make_double2(0.0, 0.0);
      if (GENERAL) {
        w2 = *reinterpret_cast<const double2*>(sw + j0 + 2 * c);
        mu2 = *reinterpret_cast<const double2*>(smu + j0 + 2 * c);
      }
      double2 x2;
#pragma unroll
      for (int hlf = 1; hlf >= 0; --hlf) {
        const int k = 2 * c + hlf;
        const double pdk = hlf ? pd2.y : pd2.x, pek = hlf ? pe2.y : pe2.x, yk = hlf ? y2.y : y2.x;
        const double wk = hlf ? w2.y : w2.x, muk = hlf ? mu2.y : mu2.x;
        const double x = fma(-m[k], xn, g[k]);
        const double r = GENERAL ? x - muk : x;
        if (k < nvalid) {
          ssp = fma(pdk * r, r, ssp);
          ssp2 = fma(pek * r, rn, ssp2);
          const double q = yk - x;
          ssl = GENERAL ? fma(wk * q, q, ssl) : fma(q, q, ssl);
        }
        if (hlf) x2.y = x; else x2.x = x;
        xn = x;
        rn = r;
      }
      *reinterpret_cast<double2*>(sy + j0 + 2 * c) = x2;
    }
    bulk_out = (i_t + TG_TILE <= n) && al16(a.x + (long long)chain * n + i_t);
    if (bulk_out) asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
  }
  // ---- per-tile partial sums (fixed order: shuffle tree, then the 4 warps in order)
  ssp = omc_warp_sum(fma(2.0, ssp2, ssp));
  ssl = omc_warp_sum(ssl);
  if (DEBUG) logdet = omc_warp_sum(logdet);
  if (lane == 0) {
    s_part[warp] = ssp;
    s_part[TG_NW + warp] = ssl;
    s_part[2 * TG_NW + warp] = logdet;
  }
  __syncthreads();
  if (solve) {   // x tile: shared -> global (one bulk store for full aligned tiles)
    double* xg = a.x + (long long)chain * n + i_t;
    if (bulk_out) {
      if (tid == 0) bulk_s2g(xg, sy, TG_TILE * 8);
    } else {
      for (int j = tid; j < TG_TILE; j += TG_NT)
        if (i_t + j < n) xg[j] = sy[j];
    }
  }
  if (tid == 0) {   // per-tile partials; tg_partials_kernel reduces them per chain in a fixed order
    double sp = 0.0, sl = 0.0, ld = 0.0;
    for (int w = 0; w < TG_NW; ++w) { sp += s_part[w]; sl += s_part[TG_NW + w]; ld += s_part[2 * TG_NW + w]; }
    *reinterpret_cast<double2*>(parts) = make_double2(sp, sl);
    parts[2] = ld;
    if (s_bad && a.status) atomicOr(&a.status[chain], OMC_STATUS_NOT_PD);
    if (solve && bulk_out) bulk_store_wait();   // shared memory must stay alive until the bulk store has read it
  }
}

// Per-chain sums of the per-tile partials, fixed order (deterministic): one warp per chain.
__global__ void __launch_bounds__(32) tg_partials_kernel(Workspace* ws, Layout L, long long n_parts, int C, double* ss_prior,
                                                          double* ss_lik, double* logdet) {
  const int chain = blockIdx.x, lane = threadIdx.x;
  const double* parts = reinterpret_cast<const double*>(reinterpret_cast<char*>(ws) + L.off_parts);
  double sp = 0.0, sl = 0.0, ld = 0.0;
  for (long long t = lane; t < n_parts; t += 32) {
    const double* p = parts + (t * C + chain) * 4;
    const double2 v = *reinterpret_cast<const double2*>(p);
    sp += v.x;
    sl += v.y;
    if (logdet) ld += p[2];
  }
  sp = omc_warp_sum(sp);
  sl = omc_warp_sum(sl);
  ld = omc_warp_sum(ld);
  if (lane == 0) {
    if (ss_prior) ss_prior[chain] = sp;
    if (ss_lik) ss_lik[chain] = sl;
    if (logdet) logdet[chain] = ld;
  }
}

// ---------------------------------------------------------------------------------------------- quadratic forms only
// ss_prior = (x-mu0)' P (x-mu0), ss_lik = (y-x)' W (y-x) of the CURRENT x (ref: sampler.py:275-284); coalesced sweep,
// per-tile partials reduced per chain in a fixed order (deterministic).
__global__ void __launch_bounds__(TG_NT) tg_quadforms_kernel(omc_tridiag_nn_t a, Workspace* ws, Layout L) {
  __shared__ double s_red[2 * TG_NW];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int C = a.n_chains;
  const long long tile = blockIdx.x / C;
  const int chain = (int)(blockIdx.x % C);
  const long long n = a.n;
  char* wsb = reinterpret_cast<char*>(ws);
  double* parts = reinterpret_cast<double*>(wsb + L.off_parts) + (tile * C + chain) * 4;
  const double* xg = a.x + (long long)chain * n;
  const double* mup = a.mu0.ptr ? a.mu0.ptr + (long long)chain * a.mu0.chain_stride : nullptr;
  const double* yp = a.y.ptr ? a.y.ptr + (long long)chain * a.y.chain_stride : nullptr;
  const double* wp = a.w.ptr ? a.w.ptr + (long long)chain * a.w.chain_stride : nullptr;
  double ssp = 0.0, ssl = 0.0;
  for (int r = 0; r < TG_K; ++r) {
    const long long i = tile * TG_TILE + r * TG_NT + tid;
    if (i < n) {
      const double x = xg[i];
      const double ri = x - (mup ? __ldg(mup + i) : 0.0);
      double rn = 0.0, pe = 0.0;
      if (i + 1 < n) {
        rn = xg[i + 1] - (mup ? __ldg(mup + i + 1) : 0.0);
        pe = a.pe ? __ldg(a.pe + i) : 0.0;
      }
      ssp = fma(__ldg(a.pd + i) * ri, ri, fma(2.0 * pe * ri, rn, ssp));
      if (yp) {
        const double q = __ldg(yp + i) - x;
        ssl = fma((wp ? __ldg(wp + i) : 1.0) * q, q, ssl);
      }
    }
  }
  ssp = omc_warp_sum(ssp);
  ssl = omc_warp_sum(ssl);
  if (lane == 0) { s_red[warp] = ssp; s_red[TG_NW + warp] = ssl; }
  __syncthreads();
  if (tid == 0) {
    double sp = 0.0, sl = 0.0;
    for (int w = 0; w < TG_NW; ++w) { sp += s_red[w]; sl += s_red[TG_NW + w]; }
    *reinterpret_cast<double2*>(parts) = make_double2(sp, sl);
  }
}

__global__ void tridiag_ws_init_kernel(Workspace* ws, Layout L) {
  // zero the header and every tile record (flags)
  const long long words = L.off_flags_end / 8;
  unsigned long long* p = reinterpret_cast<unsigned long long*>(ws);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < words; i += (long long)gridDim.x * blockDim.x)
    p[i] = 0ull;
}

// Q = L L' of a lower bidiagonal factor (diagonal l, sub-diagonal c): Q_ii = l_i^2 + c_{i-1}^2, Q_{i+1,i} = c_i l_i.
// For the gmrf functions that are handed a precomputed sparse factor (gmrf.py:29-61, 167-198, 437-462).
__global__ void bidiag_gram_kernel(const double* __restrict__ l, const double* __restrict__ c, long long n,
                                   double* __restrict__ pd, double* __restrict__ pe) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const double li = l[i], cp = i > 0 ? c[i - 1] : 0.0;
    pd[i] = fma(li, li, cp * cp);
    if (i < n - 1) pe[i] = c[i] * li;
  }
}

__global__ void tridiag_matvec_kernel(const double* pd, const double* pe, omc_vec_t v, int n_chains, long long n,
                                      double* out) {
  const long long total = (long long)n_chains * n;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const int chain = (int)(t / n);
    const long long i = t % n;
    const double* vp = v.ptr + (long long)chain * v.chain_stride;
    double s = pd[i] * vp[i];
    if (i > 0) s += pe[i - 1] * vp[i - 1];
    if (i + 1 < n) s += pe[i] * vp[i + 1];
    out[t] = s;
  }
}

int check_args(const omc_tridiag_nn_t* a, const char* who) {
  OMC_REQUIRE(a && a->pd && a->workspace, "%s: null argument", who);
  OMC_REQUIRE(a->n_chains >= 1 && a->n >= 1, "%s: n_chains=%d n=%lld", who, a->n_chains, a->n);
  OMC_REQUIRE((long long)a->n_chains * ((a->n + TG_TILE - 1) / TG_TILE) < 0x7fffffffll, "%s: too many tiles", who);
  return 0;
}

constexpr int aggregate_smem_doubles(bool general, int g) { return 4 + (general ? 5 : 2 + g) * TG_TILE + 4; }
constexpr int solve_smem_doubles(bool general, bool debug) {
  return 4 + (3 + (debug ? 1 : 0) + (general ? 3 : 0)) * TG_TILE + 4;
}

template <bool GENERAL, int G>
int launch_aggregate(const omc_tridiag_nn_t& a, Workspace* ws, const Layout& L, cudaStream_t st) {
  const int smem = aggregate_smem_doubles(GENERAL, G) * 8;
  const int n_groups = (a.n_chains + G - 1) / G;
  OMC_CHECK_CUDA(cudaFuncSetAttribute(tg_aggregate_kernel<GENERAL, G>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  tg_aggregate_kernel<GENERAL, G><<<(unsigned int)(L.n_tiles * n_groups), TG_NT * G, smem, st>>>(a, ws, L, n_groups);
  OMC_LAUNCH_CHECK();
  return 0;
}
template <bool GENERAL, bool DEBUG>
int launch_solve(const omc_tridiag_nn_t& a, Workspace* ws, const Layout& L, unsigned grid, cudaStream_t st) {
  const int smem = solve_smem_doubles(GENERAL, DEBUG) * 8;
  OMC_CHECK_CUDA(cudaFuncSetAttribute(tg_solve_kernel<GENERAL, DEBUG>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  tg_solve_kernel<GENERAL, DEBUG><<<grid, TG_NT, smem, st>>>(a, ws, L);
  OMC_LAUNCH_CHECK();
  return 0;
}

}  // namespace

extern "C" {

int omc_tridiag_workspace(int n_chains, long long n, long long* bytes) {
  OMC_REQUIRE(n_chains >= 1 && n >= 1 && bytes, "omc_tridiag_workspace: bad argument");
  *bytes = make_layout(n_chains, n).total;
  return 0;
}

int omc_tridiag_workspace_init(void* workspace, int n_chains, long long n, void* stream) {
  OMC_REQUIRE(workspace, "omc_tridiag_workspace_init: null workspace");
  const Layout L = make_layout(n_chains, n);
  tridiag_ws_init_kernel<<<256, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<Workspace*>(workspace), L);
  OMC_LAUNCH_CHECK();
  return 0;
}

int omc_tridiag_nn_draw(const omc_tridiag_nn_t* a, void* stream) {
  if (a) OMC_REQUIRE_SITE(a->rng, "omc_tridiag_nn_draw");
  if (int rc = check_args(a, "omc_tridiag_nn_draw")) return rc;
  OMC_REQUIRE(a->y.ptr, "omc_tridiag_nn_draw: y missing");
  const Layout L = make_layout(a->n_chains, a->n);
  const unsigned int grid = (unsigned int)(L.n_tiles * a->n_chains);
  Workspace* ws = reinterpret_cast<Workspace*>(a->workspace);
  cudaStream_t st = (cudaStream_t)stream;
  const bool general = a->w.ptr || a->h.ptr || a->mu0.ptr;
  const bool debug = a->debug_z || a->logdet || a->probe_l || a->probe_c || !a->x;
  int rc;
  if (general) rc = launch_aggregate<true, 1>(*a, ws, L, st);
  else if (a->n_chains >= TG_AGG_G) rc = launch_aggregate<false, TG_AGG_G>(*a, ws, L, st);
  else rc = launch_aggregate<false, 1>(*a, ws, L, st);
  if (rc) return rc;
  tg_tilescan_kernel<<<a->n_chains, TS_NT, 0, st>>>(ws, L, a->n_chains);
  OMC_LAUNCH_CHECK();
  if (general) rc = debug ? launch_solve<true, true>(*a, ws, L, grid, st) : launch_solve<true, false>(*a, ws, L, grid, st);
  else rc = debug ? launch_solve<false, true>(*a, ws, L, grid, st) : launch_solve<false, false>(*a, ws, L, grid, st);
  if (rc) return rc;
  const bool solve = a->x != nullptr;
  if ((solve && (a->ss_prior || a->ss_lik)) || a->logdet) {
    tg_partials_kernel<<<a->n_chains, 32, 0, st>>>(ws, L, L.n_tiles, a->n_chains, solve ? a->ss_prior : nullptr,
                                                   solve ? a->ss_lik : nullptr, a->logdet);
    OMC_LAUNCH_CHECK();
  }
  return 0;
}

int omc_tridiag_quadforms(const omc_tridiag_nn_t* a, void* stream) {
  if (int rc = check_args(a, "omc_tridiag_quadforms")) return rc;
  OMC_REQUIRE(a->x, "omc_tridiag_quadforms: x missing");
  const Layout L = make_layout(a->n_chains, a->n);
  const unsigned int grid = (unsigned int)(L.n_tiles * a->n_chains);
  Workspace* ws = reinterpret_cast<Workspace*>(a->workspace);
  tg_quadforms_kernel<<<grid, TG_NT, 0, (cudaStream_t)stream>>>(*a, ws, L);
  OMC_LAUNCH_CHECK();
  tg_partials_kernel<<<a->n_chains, 32, 0, (cudaStream_t)stream>>>(ws, L, L.n_tiles, a->n_chains, a->ss_prior, a->ss_lik,
                                                                    nullptr);
  OMC_LAUNCH_CHECK();
  return 0;
}

int omc_bidiag_gram(const double* l, const double* c, long long n, double* pd, double* pe, void* stream) {
  OMC_REQUIRE(l && pd && n >= 1 && (n == 1 || (c && pe)), "omc_bidiag_gram: bad argument");
  const unsigned int blocks = (unsigned int)((n + 255) / 256 > 148 * 16 ? 148 * 16 : (n + 255) / 256);
  bidiag_gram_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(l, c, n, pd, pe);
  OMC_LAUNCH_CHECK();
  return 0;
}

int omc_tridiag_matvec(const double* pd, const double* pe, omc_vec_t v, int n_chains, long long n, double* out,
                       void* stream) {
  OMC_REQUIRE(pd && v.ptr && out && n_chains >= 1 && n >= 1 && (n == 1 || pe), "omc_tridiag_matvec: bad argument");
  const long long total = (long long)n_chains * n;
  const unsigned int blocks = (unsigned int)((total + 255) / 256 > 148 * 16 ? 148 * 16 : (total + 255) / 256);
  tridiag_matvec_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(pd, pe, v, n_chains, n, out);
  OMC_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
