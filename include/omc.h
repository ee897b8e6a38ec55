/* libomc — C ABI of the B200-native openMCMC hot path.
 *
 * The reference (sede-open/openMCMC, pure Python) has no FFI boundary; its seam is the duck-typed sampler / model
 * interface that mcmc.MCMC calls (SURVEY.md §8b).  This header is the boundary a maintainer would bind from
 * Python (ctypes stub in INTEGRATION.md): every entry point below names the reference code it replaces as
 * `ref: <file>:<lines>` relative to /root/reference/src/openmcmc/.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host; all reals are float64 (the reference is fp64)
 *   - `void* stream` is a cudaStream_t (0 = legacy default stream); every call is asynchronous on that stream
 *   - omc_vec_t = per-chain operand: element c lives at ptr + c*chain_stride; chain_stride 0 = shared by all chains;
 *     ptr NULL = the documented default
 *   - return 0 = ok, <0 = argument / plan error, >0 = cudaError_t; text via omc_last_error() (thread local)
 *   - numerical failures never abort a batch: they set bits in the per-chain `status` word (OMC_STATUS_*)
 *   - ownership: the caller owns every buffer; the library owns only what omc_*_create returns
 */
#ifndef OMC_H
#define OMC_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define OMC_ABI_VERSION 1
#define OMC_STATUS_NOT_PD 1          /* Cholesky pivot <= 0 (reference: LinAlgError from np.linalg.cholesky) */
#define OMC_STATUS_NAN 2             /* NaN/inf in the log-density or gradient of the CURRENT state            */
#define OMC_STATUS_OUT_OF_SUPPORT 4  /* a PROPOSAL was invalid (outside the support / non-PD Hessian) and was
                                        rejected; informational (the reference crashes here, SURVEY F6)         */

typedef struct {
  const double* ptr;
  long long chain_stride;
} omc_vec_t;

/* Counter-based RNG site (Philox4x32-10).  Replaces the reference's global numpy RandomState reached through
 * scipy.stats.*.rvs (SURVEY F7).  Draw = f(seed, sweep counter, global chain id, site, position). */
typedef struct {
  unsigned long long seed;
  const unsigned long long* sweep; /* device counter, bumped once per sweep (omc_counter_add); NULL = 0 */
  unsigned int chain_offset;       /* global id of local chain 0 (multi-GPU sharding)                  */
  unsigned int site;               /* one id per sampler in the plan                                    */
} omc_rng_t;

/* ------------------------------------------------------------------ library / device */
int omc_abi_version(void);
const char* omc_last_error(void);
int omc_device_init(int device);          /* cudaSetDevice + attribute cache; must precede everything else */
int omc_device_sm_count(void);
int omc_counter_add(unsigned long long* counter, unsigned long long inc, void* stream);
/* both counters of a stored sweep (sweep counter, stored-iteration counter) in one launch */
int omc_counter_add2(unsigned long long* c0, unsigned long long inc0, unsigned long long* c1, unsigned long long inc1,
                     void* stream);

/* ------------------------------------------------------------------ sweep execution (ref: mcmc.py:87-111)
 * A sweep is recorded once as a CUDA graph (capture between begin/end on `stream`, calling the op entry points
 * below) and replayed by omc_run_schedule with the reference's iteration numbering: (n_burn+n_iter) outer
 * iterations of n_thin sweeps; after each non-burn iteration the `store` graph runs once. */
typedef struct omc_graph omc_graph_t;
int omc_graph_capture_begin(void* stream);
int omc_graph_capture_end(void* stream, omc_graph_t** out);
int omc_graph_launch(omc_graph_t* g, void* stream, long long times);
int omc_graph_destroy(omc_graph_t* g);
int omc_graph_num_kernel_nodes(omc_graph_t* g, long long* out);
int omc_run_schedule(omc_graph_t* sweep, omc_graph_t* store, void* stream, long long n_burn, long long n_iter,
                     long long n_thin);
/* store[iter] <- src : `count` doubles into dst + (*iter_counter)*count   (ref: sampler.py:89-118) */
int omc_store_copy(const double* src, double* dst, long long count, const unsigned long long* iter_counter,
                   long long max_iter, void* stream);
/* streamed store: slab (*iter_counter % ring) of a device ring [ring][count]; the host drains slab k to pinned memory on
 * a copy stream while the sweeps of the next stored iterations run (north star: "samples stream asynchronously to
 * pinned host memory"; ref: mcmc.py:105-111, sampler.py:89-118) */
int omc_store_copy_ring(const double* src, double* dst, long long count, const unsigned long long* iter_counter,
                        long long ring, void* stream);

/* ------------------------------------------------------------------ conjugate regression (C1 / C2)
 * omc_reg_pass: one fused pass over (X, y[, w]) per chain -> record  G = X'WX | g = X'Wy | rss | cnt
 *   ref: location_scale.py:234-242 (Hessian X'QX), sampler.py:190-192 (X'Q(y-d)), sampler.py:275-284 (r'Pr, #diag>0)
 *   X: [n x p] row-major per chain; y,w: [n]; beta: [p] (NULL => rss = y'Wy); stats: [n_chains][p*p+p+2]
 *   workspace: omc_reg_pass_workspace() doubles when n_split > 1 (few chains, long n), else may be NULL. */
int omc_reg_pass_workspace(int n_chains, int n, int p, int* n_split_out, long long* workspace_doubles);
int omc_reg_pass(const double* X, long long strideX, const double* y, long long strideY, const double* w,
                 long long strideW, const double* beta, long long strideB, int n_chains, int n, int p,
                 double* stats, double* workspace, void* stream);
/* omc_reg_rss: the residual-only pass.  rss = (y - X beta)' W (y - X beta) and cnt are written into the same record;
 *   G and g are left as they are: they depend on the data alone, so a Gibbs sweep whose likelihood weights are not
 *   sampled keeps them from one omc_reg_pass in the prologue and streams X once per sweep for the residual only
 *   (HBM-bound, no tensor work).  Same arguments as omc_reg_pass; beta must not be NULL.
 *   ref: sampler.py:275-284 (residual.T @ P @ residual of NormalGamma.sample), mcmc.py:108 (log_post) */
int omc_reg_rss(const double* X, long long strideX, const double* y, long long strideY, const double* w,
                long long strideW, const double* beta, long long strideB, int n_chains, int n, int p,
                double* stats, double* workspace, void* stream);

/* omc_nn_dense_draw: NormalNormal conditional draw for a dense p x p posterior precision (p <= 512; p <= 32 one
 *   thread per column in registers, above that a blocked Cholesky with a DMMA trailing update)
 *   Q = lambda*P0 + tau*G ; b = lambda*P0*mu0 + tau*g ; L = chol(Q) ; mu = L^-T L^-1 b ; beta = mu + L^-T z
 *   ref: sampler.py:154-207 (NormalNormal.sample), gmrf.py:167-198 (sample_normal_canonical), gmrf.py:29-61 */
typedef struct {
  int n_chains, p;
  omc_vec_t stats;      /* records from omc_reg_pass (chain_stride = p*p+p+2)                */
  omc_vec_t tau;        /* scalar multiplying G and g; NULL => 1                             */
  int prior_kind;       /* 0 scaled identity, 1 diagonal, 2 dense row-major                  */
  omc_vec_t prior_P;    /* un-scaled prior precision (kind 0: 1 value or NULL => 1)          */
  omc_vec_t lambda;     /* scalar multiplying prior_P; NULL => 1                             */
  omc_vec_t mu0;        /* prior mean [p]; NULL => 0                                         */
  double* beta;         /* out [n_chains][p]                                                 */
  omc_rng_t rng;
  const double* debug_z; /* injected standard normals [n_chains][p] (ref tests patch norm.rvs); NULL => Philox */
  long long debug_sweep_stride; /* elements between consecutive sweeps' injected draws (0 = same every sweep) */
  double* probe_Q;      /* optional [n_chains][p*p] posterior precision                      */
  double* probe_b;      /* optional [n_chains][p]                                            */
  double* probe_L;      /* optional [n_chains][p*p] lower Cholesky factor                    */
  double* probe_mu;     /* optional [n_chains][p] posterior mean                             */
  int* status;          /* optional [n_chains], OR-ed with OMC_STATUS_*                      */
  /* Truncated prior (domain_response_lower / upper on the Normal prior): the draw becomes ONE coordinate-wise Gibbs
   * scan from the current beta,  beta_i ~ N(v_i (b_i - Q_i. beta + Q_ii beta_i), v_i = 1/Q_ii) truncated to
   * [lo_i, hi_i], one truncnorm.rvs uniform per coordinate (Philox block i of the chain, or debug_u); p == 1 draws
   * from N(b/Q, 1/Q) truncated.  p <= 64: Q in shared memory, one CTA per chain; 64 < p <= 512: one warp per chain
   * streaming the rows of G (and of a dense P0) through shared memory; p > 512 is refused.  probe_Q / probe_b are
   * written; center, rss_out, mode and workspace are ignored.
   *   ref: sampler.py:196-205, gmrf.py:201-266 (gibbs_canonical_truncated_normal), gmrf.py:269-292 */
  int truncated;        /* 0: plain draw above (trunc_* ignored)                             */
  omc_vec_t trunc_lo, trunc_hi; /* bounds, trunc_lo_len / trunc_hi_len in {1, p} values (NULL => -inf / +inf) */
  int trunc_lo_len, trunc_hi_len;
  const double* debug_u; /* injected uniforms behind truncnorm.rvs [n_chains][p]; NULL => Philox; strided by
                            debug_sweep_stride like debug_z                                   */
  /* Re-centred sufficient statistics: with the per-chain centre record  beta_hat [p] | c0 = X'W(y - X beta_hat) [p] |
   * rss0 = (y - X beta_hat)'W(y - X beta_hat)  (chain_stride >= 2p+1) the draw also writes
   *   rss(beta) = rss0 - 2 d'c0 + d'G d,  d = beta - beta_hat,
   * to rss_out[chain * stats.chain_stride]: the residual sum of squares NormalGamma.sample and log_post need
   * (sampler.py:275-284, mcmc.py:108) without a pass over X.  No cancellation when beta_hat is the least-squares
   * point (c0 ~ 0, both remaining terms >= 0).  NULL => not written. */
  omc_vec_t center;
  double* rss_out;
  int mode;             /* 0: draw; 1: solve only: beta = (Q with diag *= 1 + ridge_rel)^-1 b, no z, no status bit (a
                           non-PD matrix gives beta = 0): how the prologue gets the centre beta_hat              */
  double ridge_rel;
  double* workspace;    /* p above the shared-memory limit (see omc_nn_dense_workspace): scratch for the factor   */
} omc_nn_dense_t;
int omc_nn_dense_draw(const omc_nn_dense_t* args, void* stream);
/* doubles of workspace omc_nn_dense_draw / omc_dense_factor need for n_chains matrices of size p (0 while the augmented
 * matrix fits in shared memory, p <= 136) */
int omc_nn_dense_workspace(int n_chains, int p, long long* doubles);

/* omc_dense_factor: stand-alone dense SPD factorisation and solves, one CTA per matrix (n <= 512), the blocked Cholesky
 * with the DMMA trailing update that omc_nn_dense_draw runs:
 *   L = chol(Q)                              ref: gmrf.py:465-486 (cholesky), 489-520 (sparse_cholesky, dense branch)
 *   logdet = 2 sum log L_jj                  ref: gmrf.py:321-348 (multivariate_normal_pdf)
 *   mean = L^-T L^-1 b                       ref: gmrf.py:437-462 (cho_solve)
 *   x = mean + L^-T z                        ref: gmrf.py:167-198 (sample_normal_canonical), 29-61 (sample_normal),
 *                                                 414-434 (solve(L.T, z): b = NULL)
 *   factored = 1: Q already holds a lower Cholesky factor L (gmrf functions that accept a precomputed L)
 *   backward_only = 1: mean = L^-T b (no forward solve); 2: mean = L^-1 b (forward solve only), x = mean + z
 *   ref: gmrf.py:414-434 (solve with a triangular matrix: a = L' or a = L) */
typedef struct {
  int n_mats, n;
  const double* Q;      /* [n_mats][n*n] row-major (lower triangle read), matrices Q_stride doubles apart (0 = shared) */
  long long Q_stride;
  const double* b;      /* optional [n_mats][n] */
  const double* z;      /* optional [n_mats][n] */
  double* L;            /* optional out [n_mats][n*n] lower factor, zeros above the diagonal */
  double* logdet;       /* optional out [n_mats] */
  double* mean;         /* optional out [n_mats][n] */
  double* x;            /* optional out [n_mats][n] */
  int* status;          /* optional [n_mats], OR-ed with OMC_STATUS_NOT_PD */
  int factored, backward_only;
  double* workspace;    /* omc_nn_dense_workspace(n_mats, n) doubles when that is > 0 */
} omc_dense_factor_t;
int omc_dense_factor(const omc_dense_factor_t* args, void* stream);

/* omc_quadform: ss = (x-mu)' P (x-mu), cnt = #(diag P > 0) per chain  (ref: sampler.py:276-284 for a prior precision) */
typedef struct {
  int n_chains, p;
  omc_vec_t x, mu;      /* mu NULL => 0 */
  int kind;
  omc_vec_t P;
  double* ss;           /* out [n_chains] */
  double* cnt;          /* out [n_chains] */
} omc_quadform_t;
int omc_quadform(const omc_quadform_t* args, void* stream);

/* omc_ng_draw: NormalGamma conditional draw  x ~ Gamma(a0 + cnt/2, rate = b0 + ss/2)
 *   ref: sampler.py:252-288 (b == 0 => scale = inf => sample = inf guard at :285-286) */
typedef struct {
  int n_chains;
  omc_vec_t a0, b0;     /* Gamma prior shape / rate */
  omc_vec_t ss, cnt;    /* quadratic form and count (e.g. into an omc_reg_pass record) */
  double* out;          /* [n_chains] */
  omc_rng_t rng;
  const double* debug_g; /* injected standard-gamma variates Gamma(a*,1) [n_chains]; NULL => Marsaglia-Tsang */
  long long debug_sweep_stride;
  double* probe_a;      /* optional [n_chains] posterior shape */
  double* probe_b;      /* optional [n_chains] posterior rate  */
  /* vector-valued precision (the K-loop of sampler.py:281-284 over mixture components): n_elem draws per chain,
   * element k reads a0[k or 0], b0[k or 0], ss[k*ss_stride], cnt[k*cnt_stride]; out / debug_g / probes are
   * [n_chains][n_elem].  n_elem == 0 means 1 (the scalar update above). */
  int n_elem, a0_len, b0_len;
  long long ss_stride, cnt_stride;
} omc_ng_draw_t;
int omc_ng_draw(const omc_ng_draw_t* args, void* stream);

/* ------------------------------------------------------------------ mixture models (SURVEY §8 f2)
 * x_i ~ N(mu[z_i], 1/tau[z_i]), z_i ~ Categorical(prob), i < n, K components; allocations are float64 integers.
 * omc_mixture_allocation: z_i = #{k : U_i > cumsum_k(gam)}, gam_k = prob_k N(x_i; mu_k, 1/tau_k) normalised
 *   ref: sampler.py:292-355 (MixtureAllocation.sample)
 * omc_mixture_stats: per component  n_k, sum_{z_i=k} x_i, sum_{z_i=k} (x_i - mu_k)^2  (what the NormalGamma K-loop,
 *   sampler.py:272-288 with parameter.py:522-538, and a NormalNormal update of mu need); optionally the same numbers as
 *   a regression-format record  G = diag(tau_k n_k) | g = tau_k sum x | rss = sum_k tau_k S2_k | cnt = n  for
 *   omc_nn_dense_draw, the gathers mu[z_i] / tau[z_i] (MixtureParameterVector / Matrix predictors, parameter.py:437-446,
 *   494-504) and the Normal log-density of x, 0.5 (sum_k n_k log tau_k - n log 2 pi - sum_k tau_k S2_k). */
typedef struct {
  int n_chains, n, K;
  omc_vec_t x;            /* [n]                                     */
  omc_vec_t mu, tau;      /* [K]                                     */
  omc_vec_t prob;         /* [prob_rows][K], prob_rows in {1, n}     */
  int prob_rows;
  double* z;              /* [n_chains][n] out                       */
  omc_rng_t rng;
  const double* debug_u;  /* injected uniforms [n_chains][n] (the reference's uniform.rvs(size=(n,1))) */
  long long debug_sweep_stride;
} omc_mixture_alloc_t;
int omc_mixture_allocation(const omc_mixture_alloc_t* args, void* stream);
typedef struct {
  int n_chains, n, K;
  omc_vec_t x, mu, tau;
  const double* z;        /* [n_chains][n]                           */
  double* stats;          /* out [n_chains][K][4]: n_k, sum x, sum (x - mu_k)^2, 0 */
  double* record;         /* optional out [n_chains][K*K + K + 2]    */
  double* gather_mu;      /* optional out [n_chains][n]              */
  double* gather_tau;     /* optional out [n_chains][n]              */
  double* logp;           /* optional out [n_chains]                 */
  int accumulate;
} omc_mixture_stats_t;
int omc_mixture_stats(const omc_mixture_stats_t* args, void* stream);
/* out[c] (+)= sum_i log prob[i or 0][z_i]   (ref: distribution.py:318-345, multinomial(n = 1) log-pmf) */
int omc_logp_categorical(int n_chains, int n, int K, const double* z, omc_vec_t prob, int prob_rows, double* out,
                         int accumulate, void* stream);

/* ------------------------------------------------------------------ log-densities (ref: Model.log_p, model.py:57-70)
 * Every kernel writes out[c] (accumulate = 0) or adds to it (accumulate = 1), one value per chain. */

/* Normal log-pdf from a pre-computed quadratic form with the UN-scaled precision matrix P:
 *   0.5 * (dim*log(scalar) + logdet(P) - dim*log(2 pi) - scalar*ss)
 * ref: location_scale.py:145-167 -> gmrf.py:321-348 (the reference re-factorises scalar*P on every call; log|scalar*P|
 * = dim*log(scalar) + log|P| with log|P| computed once for a constant P). */
typedef struct {
  int n_chains;
  double dim;
  omc_vec_t ss;       /* r' P r                                  */
  omc_vec_t scalar;   /* NULL => 1                               */
  omc_vec_t logdet;   /* log|P|, NULL => 0 (identity)            */
  double* out;
  int accumulate;
} omc_logp_normal_ss_t;
int omc_logp_normal_ss(const omc_logp_normal_ss_t* args, void* stream);

/* Gamma(shape, rate) log-pdf summed over n_elem responses per chain, scipy.stats.gamma.logpdf semantics:
 *   xlogy(a-1, x/scale) - x/scale - gammaln(a) - log(scale), scale = 1/rate; -inf for x < 0
 * ref: distribution.py:241-261.  shape / rate hold shape_len / rate_len (1 or n_elem) values per chain. */
typedef struct {
  int n_chains, n_elem, shape_len, rate_len;
  omc_vec_t x, shape, rate;
  double* out;
  int accumulate;
} omc_logp_gamma_t;
int omc_logp_gamma(const omc_logp_gamma_t* args, void* stream);

/* Poisson(rate) log-pmf summed over n_elem responses: xlogy(k, mu) - gammaln(k+1) - mu; -inf for k<0 or non-integer k
 * ref: distribution.py:490-508 */
typedef struct {
  int n_chains, n_elem, rate_len;
  omc_vec_t k, rate;
  double* out;
  int accumulate;
} omc_logp_poisson_t;
int omc_logp_poisson(const omc_logp_poisson_t* args, void* stream);

/* out[c] (+)= value  — constant log-densities such as Uniform (ref: distribution.py:422-442) */
int omc_logp_const(double value, int n_chains, double* out, int accumulate, void* stream);

/* out[c] += -inf when any of the n_elem values x[c] lies outside [lower, upper] (bounds: lo_len / hi_len in {1, n_elem}
 * values, NULL => unbounded): the domain test of a truncated Normal, whose log_p ignores the truncation normaliser
 * ref: location_scale.py:148-151,164-165 */
int omc_logp_domain(int n_chains, int n_elem, omc_vec_t x, omc_vec_t lower, int lo_len, omc_vec_t upper, int hi_len,
                    double* out, void* stream);

/* out[c][i] = sum_t scale_t[c] * x_t[c][i], t < n_terms <= 4, i < len (scale == NULL or scale_t.ptr == NULL => 1).
 *   - ScaledMatrix.predictor: scalar * matrix (ref: parameter.py:319-329), one "chain", the matrix values as x_0
 *   - NormalNormal with several likelihood terms: the records tau_l * (G_l | g_l) summed into one (ref: sampler.py:179-192,
 *     Q += Q_dist, b += A' Q_rsp (y - d) for every distribution of the conditional model) */
int omc_combine(int n_chains, long long len, int n_terms, const omc_vec_t* x, const omc_vec_t* scale, double* out,
                void* stream);

/* omc_fused_small: up to OMC_FUSED_MAX_OPS of the per-chain O(1) / O(p) operations above in ONE launch, executed in
 * order by the thread that owns the chain (their dependencies are per chain: e.g. the Gamma draw of tau reads the rss
 * of its own chain).  A Gibbs sweep of the regression model is the draw kernel + one fused launch (Gamma draws,
 * quadratic form) + the counter; its store epilogue (sample copies, the log-density terms of mcmc.py:108, the log_post
 * copy) is one more.  Launch-bound sweeps (C1, C4) spend most of their time between kernels otherwise.
 *   kinds: the argument structs of omc_logp_normal_ss / omc_logp_gamma / omc_logp_poisson / omc_logp_const /
 *          omc_ng_draw / omc_quadform (scaled-identity and diagonal P) / omc_store_copy(_ring)
 *   store copies are spread over all threads of the grid (coalesced); a copy whose source is produced by an earlier op
 *   of the same launch must have count == n_chains (element c is then copied by the thread of chain c). */
#define OMC_FUSED_MAX_OPS 12
enum { OMC_FOP_LOGP_NORMAL_SS = 1, OMC_FOP_LOGP_GAMMA = 2, OMC_FOP_LOGP_POISSON = 3, OMC_FOP_LOGP_CONST = 4,
       OMC_FOP_NG_DRAW = 5, OMC_FOP_QUADFORM = 6, OMC_FOP_STORE_COPY = 7 };
typedef struct {
  int kind;
  union {
    omc_logp_normal_ss_t normal_ss;
    omc_logp_gamma_t gamma;
    omc_logp_poisson_t poisson;
    struct { double value; double* out; int accumulate; } konst;
    omc_ng_draw_t ng;
    omc_quadform_t quad;
    struct { const double* src; double* dst; long long count; const unsigned long long* iter_counter; long long max_iter;
             int ring; } copy;
  } u;
} omc_fop_t;
typedef struct {
  int n_chains, n_ops;
  omc_fop_t ops[OMC_FUSED_MAX_OPS];
} omc_fused_small_t;
int omc_fused_small(const omc_fused_small_t* args, void* stream);

/* yhat[c] = sum_t X_t[c] @ theta_t[c] for up to 4 terms (ref: parameter.py:162-197 LinearCombination.predictor) */
typedef struct {
  int n_chains, n, n_terms;
  int p[4];
  omc_vec_t X[4];      /* [n x p_t] row-major */
  omc_vec_t theta[4];  /* [p_t]               */
  double* out;         /* [n_chains][n]       */
  int transform_exp[4]; /* term t uses exp(theta_t) (ref: parameter.py:232-297 LinearCombinationWithTransform) */
  omc_vec_t residual_of; /* optional [n]: out = residual_of - yhat, i.e. y - predictor_conditional(exclude) of
                            NormalNormal.sample for a mean with several terms (ref: sampler.py:188-192)          */
} omc_linear_predictor_t;
int omc_linear_predictor(const omc_linear_predictor_t* args, void* stream);

/* One-off helpers for CONSTANT precision matrices (data, not sampled): log-determinants used by the Normal log-pdf.
 * n_mats matrices, each `n` diagonal entries (sum_log) or an n x n dense SPD matrix, n <= 64 (logdet_dense: 2*sum log diag chol).
 * ref: gmrf.py:339-342 */
int omc_sum_log(const double* x, int n_mats, long long n, double* out, void* stream);
/* out[i] = log(x[i]): the log-response of a LogNormal whose response is data, ref: location_scale.py:296-303 */
int omc_log_elements(const double* x, long long n, double* out, void* stream);
int omc_logdet_dense(const double* P, int n_mats, int n, double* out, void* stream);

/* ------------------------------------------------------------------ temporal GMRF: tridiagonal NormalNormal (C3)
 * Posterior precision Q = lambda*P + tau*W with P tridiagonal (main pd[n], off pe[n-1], shared by all chains; the RW1
 * precision of gmrf.py:351-411) and W diagonal (w) or identity;  b = lambda*h + tau*W*y with h = P*mu0.
 * omc_tridiag_nn_draw: x = L^-T (L^-1 b + z), L = natural-order Cholesky factor of Q, plus the quadratic forms of the
 * new state  ss_prior = (x-mu0)'P(x-mu0),  ss_lik = (y-x)'W(y-x)  that the NormalGamma updates of lambda / tau need.
 *   ref: sampler.py:154-207, gmrf.py:167-198 (sample_normal_canonical), :489-520 (sparse_cholesky, natural order, no
 *        pivoting), :437-462 (cho_solve), :29-61 (sample_normal), sampler.py:275-284 (quadratic forms)
 * Parallel exact scans (pivots: Moebius maps; solves: affine maps) with decoupled look-back replace the sequential
 * recurrences; x == NULL runs the factorisation only (logdet / probes).  A pivot <= 0 sets OMC_STATUS_NOT_PD.
 * workspace: omc_tridiag_workspace() bytes, zero-filled once (omc_tridiag_workspace_init or a zeroed allocation). */
typedef struct {
  int n_chains;
  long long n;
  const double* pd;      /* [n]   main diagonal of P (shared)                                  */
  const double* pe;      /* [n-1] off diagonal of P (shared)                                   */
  omc_vec_t lambda, tau; /* scalars (NULL => 1)                                                */
  omc_vec_t w;           /* [n] diagonal of W (NULL => identity)                               */
  omc_vec_t y;           /* [n] response                                                       */
  omc_vec_t h;           /* [n] P*mu0 (NULL => 0)                                              */
  omc_vec_t mu0;         /* [n] prior mean (NULL => 0), used by the prior quadratic form       */
  double* x;             /* [n_chains][n] out (quadforms: in)                                  */
  omc_rng_t rng;
  const double* debug_z; /* injected N(0,1) [n_chains][n]; NULL => Philox                      */
  long long debug_sweep_stride;
  double* ss_prior;      /* optional out [n_chains]                                            */
  double* ss_lik;        /* optional out [n_chains]                                            */
  double* logdet;        /* optional out [n_chains]: log|Q| = sum log pivots                   */
  double* probe_l;       /* optional out [n_chains][n]   diagonal of L                         */
  double* probe_c;       /* optional out [n_chains][n-1] sub-diagonal of L                     */
  int* status;           /* optional [n_chains]                                                */
  void* workspace;
} omc_tridiag_nn_t;
int omc_tridiag_workspace(int n_chains, long long n, long long* bytes);
int omc_tridiag_workspace_init(void* workspace, int n_chains, long long n, void* stream);
int omc_tridiag_nn_draw(const omc_tridiag_nn_t* args, void* stream);
/* quadratic forms of the CURRENT x only (no draw): ss_prior / ss_lik as above (ref: sampler.py:275-284) */
int omc_tridiag_quadforms(const omc_tridiag_nn_t* args, void* stream);
/* out = P v for the shared tridiagonal P and per-chain / shared v [n]  (prior-mean term P*mu0, sampler.py:181-183) */
/* Q = L L' of a lower BIDIAGONAL factor (diagonal l [n], sub-diagonal c [n-1]) as tridiagonal diagonals pd [n], pe [n-1]:
 * the gmrf functions that accept a precomputed sparse factor (ref: gmrf.py:29-61 sample_normal(L=...), 437-462 cho_solve) */
int omc_bidiag_gram(const double* l, const double* c, long long n, double* pd, double* pe, void* stream);
int omc_tridiag_matvec(const double* pd, const double* pe, omc_vec_t v, int n_chains, long long n, double* out,
                       void* stream);

/* ------------------------------------------------------------------ Metropolis-Hastings family (C4)
 * The conditional model of the sampled parameter theta (n_elem values per chain) is a sum of up to 4 terms.
 * ref: Model.log_p / grad_log_p (model.py:57-112) over the conditional model (sampler.py:53-55). */
#define OMC_TERM_POISSON_RATE 1     /* data k ~ Poisson(rate = theta)                ref: distribution.py:490-508          */
#define OMC_TERM_GAMMA_RESPONSE 2   /* theta ~ Gamma(shape p1, rate p2)              ref: distribution.py:241-261          */
#define OMC_TERM_NORMAL_RESPONSE 3  /* theta ~ N(p1, (scalar*P)^-1), optional domain ref: location_scale.py:145-188,222-232 */
#define OMC_TERM_UNIFORM_RESPONSE 4 /* theta ~ U(p1, p2): constant log-density       ref: distribution.py:422-442          */
#define OMC_TERM_LOGNORMAL_RESPONSE 5 /* theta ~ LogNormal(p1, (scalar*P)^-1) (fields as NORMAL) ref: location_scale.py:276-418 */
#define OMC_TERM_NORMAL_LINEAR 6    /* data y ~ N(X f(theta), (scalar*W)^-1), f = identity or exp (transform_exp), W = eye or
                                       diagonal: evaluated through the data-only record  G = X'WX | g = X'Wy | y'Wy | cnt  of
                                       omc_reg_pass(beta = NULL):  S(f) = y'Wy - 2 g'f + f'G f,
                                       log p = (n_data log scalar + logdet - n_data log 2pi - scalar S)/2,
                                       grad = scalar f'(theta) o (g - G f),  H = scalar diag(f') G diag(f')
                                       ref: location_scale.py:145-167, 234-250; parameter.py:162-228, 232-297              */
typedef struct {
  int kind;
  int mat_kind;        /* NORMAL: 0 eye / 1 diag / 2 dense storage of P                         */
  int p1_len, p2_len;  /* 1 or n_elem                                                            */
  omc_vec_t data;      /* POISSON: the counts k [n_elem]                                         */
  omc_vec_t p1, p2;    /* GAMMA: shape, rate; NORMAL: p1 = mean; UNIFORM: lower, upper           */
  omc_vec_t P;         /* NORMAL: un-scaled precision                                            */
  omc_vec_t scalar;    /* NORMAL: scalar multiplying P (NULL => 1)                               */
  omc_vec_t logdet;    /* NORMAL: log|P| (NULL => 0)                                             */
  double dom_lo, dom_hi; /* NORMAL: log_p = -inf outside [dom_lo, dom_hi] (+-inf = unbounded)    */
  omc_vec_t stats;     /* NORMAL_LINEAR: regression record (chain_stride = n_elem^2 + n_elem + 2)  */
  int n_data;          /* NORMAL_LINEAR: length of the response y                                  */
  int transform_exp;   /* NORMAL_LINEAR: mean = X exp(theta) (LinearCombinationWithTransform)      */
} omc_term_t;
typedef struct {
  int n_chains, n_elem, n_terms;
  omc_term_t terms[4];
} omc_mh_model_t;

/* out[c] = sum of the terms' log-densities at theta[c]  (theta: [n_chains][n_elem]) */
int omc_mh_logp(const omc_mh_model_t* model, const double* theta, double* out, void* stream);
/* same, out[c] += ... when accumulate != 0 (log_post of distributions that have no dedicated omc_logp_* kernel) */
int omc_mh_logp_acc(const omc_mh_model_t* model, const double* theta, double* out, int accumulate, void* stream);
/* grad [n_chains][n_elem] of the POSITIVE log-density, hess [n_chains][n_elem^2] of the NEGATIVE log-density (may be NULL).
 * method 0: analytic derivatives (what the samplers use)
 * method 1: the reference's central finite differences, step 1e-4, Hessian = FD of the FD gradient, applied per term as
 *           the reference does (Normal terms stay analytic)   ref: distribution.py:124-198 */
int omc_mh_grad_hess(const omc_mh_model_t* model, const double* theta, int method, double* grad, double* hess,
                     void* stream);

/* RandomWalk (loop = 0: all elements at once) and RandomWalkLoop (loop = 1: one column of the (p_dim, n_rep) parameter
 * at a time, each with its own accept/reject).  limits != NULL => truncated-normal proposals with the asymmetric
 * proposal densities.  Accept iff log(u) < log_accept (strict; NaN rejects).
 * ref: metropolis_hastings.py:127-173 (accept), :212-269 (proposal), :276-289 (loop); gmrf.py:269-318 (truncnorm) */
typedef struct {
  omc_mh_model_t model;
  double* theta;             /* [n_chains][p_dim*n_rep] in/out, row-major (p_dim, n_rep)                 */
  int p_dim, n_rep, loop;
  omc_vec_t step;            /* step sizes; step_rows in {1,p_dim}, step_cols in {1,n_rep}              */
  int step_rows, step_cols;
  const double* limits;      /* [p_dim][2] lower, upper (shared by all chains) or NULL                  */
  omc_rng_t rng;
  const double* debug_z;     /* injected proposal variates: N(0,1) (untruncated) or the uniforms behind
                                truncnorm.rvs (truncated); [n_chains][n_steps][p_prop]                  */
  const double* debug_u;     /* injected accept uniforms [n_chains][n_steps]                            */
  long long debug_sweep_stride_z, debug_sweep_stride_u;
  long long* counters;       /* optional [n_chains][2]: accepted, proposed (ref AcceptRate)             */
  double* probe;             /* optional [n_chains][n_steps][5]: logp_cur, logp_prop, logq_fwd, logq_rev, accepted */
} omc_random_walk_t;
int omc_random_walk(const omc_random_walk_t* args, void* stream);

/* ManifoldMALA: proposal N(theta + 1/2 s^2 H^-1 g, s^2 H^-1) forward and reverse, dense H (n_elem <= 64).
 * ref: metropolis_hastings.py:292-373.  A non-PD Hessian or a NaN (proposal outside the support) REJECTS the move and
 * sets the chain's status bits; the reference raises instead (SURVEY F6). */
typedef struct {
  omc_mh_model_t model;
  double* theta;             /* [n_chains][n_elem] in/out                                               */
  double step;
  int method;                /* derivatives: 0 analytic, 1 reference finite differences                 */
  omc_rng_t rng;
  const double* debug_z;     /* injected N(0,1) [n_chains][n_elem]                                      */
  const double* debug_u;     /* injected accept uniform [n_chains]                                      */
  long long debug_sweep_stride_z, debug_sweep_stride_u;
  long long* counters;       /* optional [n_chains][2]                                                  */
  int* status;               /* optional [n_chains]                                                     */
  double* probe_mu;          /* optional [n_chains][n_elem]   forward proposal mean                     */
  double* probe_L;           /* optional [n_chains][n_elem^2] forward proposal Cholesky factor          */
  double* probe_prop;        /* optional [n_chains][n_elem]   proposed point                            */
  double* probe_scalars;     /* optional [n_chains][6]: logp_cur, logp_prop, logq_fwd, logq_rev, log_accept, accepted */
} omc_mmala_t;
int omc_mmala(const omc_mmala_t* args, void* stream);

/* element-wise truncated-normal helpers exposed for parity tests (ref: gmrf.py:269-318 / scipy.stats.truncnorm) */
int omc_truncnorm_rv(const double* mean, const double* scale, const double* lower, const double* upper,
                     const double* u, long long n, double* out, void* stream);
int omc_truncnorm_logpdf(const double* x, const double* mean, const double* scale, const double* lower,
                         const double* upper, long long n, double* out, void* stream);

/* ------------------------------------------------------------------ chain diagnostics (SURVEY §8d/e; no reference
 * counterpart: parity unpinned, numpy restatement in oracle/diagnostics.py)
 * omc_chain_stats: per chain and selected element of a stored parameter, from the device sample store
 *   samples [n_iter][n_chains][size] (written by omc_store_copy); selected elements j*elem_stride, j < n_sel.
 *   out [n_chains][n_sel][8] = n, mean, variance (n-1), ESS (autocorrelation, Geyer initial monotone sequence, lags <=
 *   min(max_lag,127)), first-half mean, first-half variance, second-half mean, second-half variance.
 * omc_rhat_combine: split-R-hat and total ESS per selected element from the records of ALL chains (every rank's
 *   records after the NCCL all-gather): out [n_sel][4] = R-hat, sum of chain ESS, grand mean, var+ . */
typedef struct {
  const double* samples;
  long long n_iter;
  int n_chains;
  long long size, n_sel, elem_stride;
  int max_lag;
  double* out;
} omc_chain_stats_t;
int omc_chain_stats(const omc_chain_stats_t* args, void* stream);
int omc_rhat_combine(const double* stats, int n_chains_total, int n_sel, double* out, void* stream);
/* Rank normalisation (Vehtari et al. 2021): z [n_iter][n_chains][n_sel] = Phi^-1((r - 3/8) / (S + 1/4)) with r the average
 * rank of the draw among the n_iter draws of its own series (pooled = 0) or among the draws of all n_chains chains of that
 * element (pooled = 1); `sorted` is scratch [n_chains][n_sel][n_iter].  omc_chain_stats / omc_rhat_combine on z give
 * bulk-ESS and rank-normalised split-R-hat.  n_iter <= 16384. */
int omc_rank_normalize(const double* samples, long long n_iter, int n_chains, long long size, long long n_sel,
                       long long elem_stride, int pooled, double* sorted, double* z, void* stream);

/* ------------------------------------------------------------------ ReversibleJump (C5)
 * One birth / death step per chain for the Gaussian-kernel basis model of the reference's RJ tests
 * (tests/test_reversible_jump.py:23-252): state of fixed capacity n_max (first n entries live), basis column
 * j = N(X; theta_j, omega_j) built in (replaces the Python state_birth/death callbacks, SURVEY F10), matched coefficient
 * transitions, move probabilities with their edge cases, accept / reject on the whole model:
 * response Normal(y | B beta, (tau_y I)^-1) or Null (y.ptr == NULL), beta ~ iid N(mu_beta, 1/tau_beta), n ~ Poisson(rho),
 * theta ~ U(theta_lo, theta_hi), omega ~ Gamma(omega_shape, omega_rate) when sample_omega.
 *   ref: sampler/reversible_jump.py:76-373; metropolis_hastings.py:127-173; gmrf.py:269-318
 * debug: injected variates per chain [6] = move uniform, new knot, new width, new coefficient (NaN => the matched mean),
 *   deletion index, accept uniform — the FINAL values of the reference's rvs calls (SURVEY B.4 order).
 * probe: [n_chains][8] = birth, deletion index, logp current, logp proposed, logq forward, logq reverse, log accept,
 *   accepted.  logp_only != 0: write the model log-density of the current state to logp_out and return. */
typedef struct {
  int n_chains, n_data, n_max;
  double* n_basis;             /* [n_chains] in/out                         */
  double* theta;               /* [n_chains][n_max] in/out                  */
  double* omega;               /* [n_chains][n_max] in/out                  */
  double* beta;                /* [n_chains][n_max] in/out                  */
  double* B;                   /* [n_chains][n_data][n_max] in/out          */
  const double* X;             /* [n_data] data locations (shared)          */
  omc_vec_t y;                 /* [n_data] response, NULL => Null response  */
  omc_vec_t tau_y;
  double theta_lo, theta_hi;
  int sample_omega;            /* 0: a new component copies the last width  */
  omc_vec_t omega_shape, omega_rate;
  omc_vec_t mu_beta, tau_beta;
  omc_vec_t rho;
  double birth_probability;
  double match_scale;
  int match_truncated;
  double match_lo, match_hi;
  omc_rng_t rng;
  const double* debug;
  long long debug_sweep_stride;
  long long* counters;         /* optional [n_chains][2]: accepted, proposed */
  int* status;                 /* optional [n_chains]                        */
  double* probe;               /* optional [n_chains][8]                     */
  int logp_only;
  double* logp_out;            /* [n_chains] when logp_only                  */
  int* size_class;             /* optional scratch [n_chains]: the step is then launched per size class of live
                                  components (small shared-memory footprint for small chains)                   */
  /* Live Gram matrix S = B'B of the current basis in the chain state (optional): [n_chains][n_max][n_max], lower
   * triangle, valid where gram_valid[c] != 0.  The matched transitions need the Gram matrix of the LARGER basis
   * (reversible_jump.py:240-242, 290-291): with it resident a birth costs the inner products of ONE new column
   * (2 n_data k flops) and a death none, instead of 2 n_data k^2 per step; an accepted move appends / deletes a row and
   * column.  Whatever rewrites basis columns (omc_rj_basis, omc_rj_knot_walk) clears gram_valid; the next step then
   * recomputes S in full and stores it. */
  double* gram;
  int* gram_valid;
} omc_rj_t;
int omc_rj_smem_bytes(int n_data, int n_max);
int omc_reversible_jump(const omc_rj_t* args, void* stream);
/* B[c][r][j] = N(X_r; theta_cj, omega_cj) for j < n_c, 0 beyond (ref: make_basis, tests/test_reversible_jump.py:23-40) */
int omc_rj_basis(const omc_rj_t* args, void* stream);

/* Companion moves of the RJ model on the same padded state (the other samplers of tests/test_reversible_jump.py:213-252).
 * omc_rj_knot_walk: RandomWalkLoop over the knots (which = 0) or widths (which = 1): per live component one truncated-
 *   Gaussian step on [lim_lo, lim_hi], basis column rebuilt for the proposal (the reference's state_update_function =
 *   make_basis), accept on the full model (only the response and the moved component's prior change).
 *   ref: metropolis_hastings.py:212-289, :127-173, :201-210; gmrf.py:269-318
 *   debug_tn_u / debug_u: injected truncnorm.rvs / accept uniforms [n_chains][n_max] (component j at index j).
 * omc_rj_coef_mmala: ManifoldMALA on the live coefficients: response Normal(y | B beta, (tau_y I)^-1) or Null, prior
 *   iid N(mu_beta, 1/tau_beta).  ref: metropolis_hastings.py:292-373, location_scale.py:222-250
 *   debug_z [n_chains][n_max], debug_u [n_chains]; probe [n_chains][6] = rss_cur, rss_prop, logq_fwd, logq_rev,
 *   log_accept, accepted.  model.size_class (optional scratch) lets chains with few live coefficients run from a small
 *   shared-memory footprint. */
typedef struct {
  omc_rj_t model;
  int which;
  double step, lim_lo, lim_hi;
  const double* debug_tn_u;
  const double* debug_u;
  long long debug_sweep_stride;
  long long* counters;         /* optional [n_chains][2]: accepted, proposed */
} omc_rj_walk_t;
int omc_rj_knot_walk(const omc_rj_walk_t* args, void* stream);
typedef struct {
  omc_rj_t model;
  double step;
  const double* debug_z;
  const double* debug_u;
  long long debug_sweep_stride_z, debug_sweep_stride_u;
  long long* counters;         /* optional [n_chains][2] */
  double* probe;               /* optional [n_chains][6] */
} omc_rj_mmala_t;
int omc_rj_coef_mmala(const omc_rj_mmala_t* args, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* OMC_H */
