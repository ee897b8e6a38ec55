"""Typed Python wrappers over the C-ABI op entry points (include/omc.h).

Device memory and streams come from torch (plumbing only); every numeric result is produced by libomc's CUDA
kernels.  Tensors are float64 CUDA tensors; per-chain operands have a leading chain dimension.
"""

import ctypes as C

import numpy as np

import torch

from openmcmc_b200 import _cabi
from openmcmc_b200._cabi import Vec, Rng, check

MAT_EYE, MAT_DIAG, MAT_DENSE = 0, 1, 2
_initialised = set()


def lib():
    return _cabi.load()


def init_device(device=None) -> int:
    """Select the CUDA device for libomc (must be sm_100a).  Raises if CUDA is unavailable — no CPU path exists."""
    if not torch.cuda.is_available():
        raise _cabi.OmcError("openmcmc_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    dev = torch.cuda.current_device() if device is None else torch.device(device).index or 0
    torch.cuda.set_device(dev)
    if dev not in _initialised:
        check(lib().omc_device_init(dev), "omc_device_init")
        _initialised.add(dev)
    return dev


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


# ----------------------------------------------------------------------------- host <-> device staging
# Pageable transfers through the driver run at ~2 GB/s on the B200 boxes and pinning a fresh multi-GB buffer costs as
# much (tools/microbench/d2h_paths.py); two persistent pinned buffers and a copy pipeline reach 15-20 GB/s into / out of
# ordinary numpy arrays.  Host plumbing only: bytes are moved, never computed on.
_STAGE_BYTES = 64 << 20
_stage = {}


def _staging(dev):
    if dev not in _stage:
        _stage[dev] = ([torch.empty(_STAGE_BYTES, dtype=torch.uint8, pin_memory=True) for _ in range(2)],
                       [torch.cuda.Event(), torch.cuda.Event()])
    return _stage[dev]


def download(t: torch.Tensor) -> np.ndarray:
    """Device tensor -> new numpy array (same shape / dtype), staged through the pinned buffers on the current stream."""
    t = t.contiguous()
    out = np.empty(tuple(t.shape), dtype=np.float64 if t.dtype == torch.float64 else
                   {torch.int32: np.int32, torch.int64: np.int64, torch.uint8: np.uint8}[t.dtype])
    nbytes = t.numel() * t.element_size()
    if nbytes == 0:
        return out
    src = t.view(-1).view(torch.uint8)
    dst = torch.from_numpy(out.reshape(-1)).view(torch.uint8)
    if nbytes <= (1 << 20):
        dst.copy_(src)           # small: one synchronous copy
        return out
    bufs, evs = _staging(t.device.index)
    pending = []
    k = 0
    for off in range(0, nbytes, _STAGE_BYTES):
        if len(pending) == 2:
            po, pb, cnt = pending.pop(0)
            evs[pb].synchronize()
            dst[po:po + cnt].copy_(bufs[pb][:cnt])
        b = k & 1
        cnt = min(_STAGE_BYTES, nbytes - off)
        bufs[b][:cnt].copy_(src[off:off + cnt], non_blocking=True)
        evs[b].record()
        pending.append((off, b, cnt))
        k += 1
    for po, pb, cnt in pending:
        evs[pb].synchronize()
        dst[po:po + cnt].copy_(bufs[pb][:cnt])
    return out


def upload(a: np.ndarray, device) -> torch.Tensor:
    """numpy array -> new device tensor through the pinned staging buffers (pinned torch tensors should be passed to
    the engine directly: they go over in one asynchronous copy)."""
    a = np.ascontiguousarray(a)
    out = torch.empty(a.shape, dtype=torch.from_numpy(a.reshape(-1)[:1]).dtype if a.size else torch.float64, device=device)
    nbytes = a.nbytes
    if nbytes <= (4 << 20):
        if nbytes:
            out.copy_(torch.from_numpy(a))
        return out
    if not a.flags.writeable:
        a = a.copy()
    src = torch.from_numpy(a.reshape(-1)).view(torch.uint8)
    dst = out.view(-1).view(torch.uint8)
    bufs, evs = _staging(out.device.index)
    k = 0
    for off in range(0, nbytes, _STAGE_BYTES):
        b = k & 1
        if k >= 2:
            evs[b].synchronize()          # the device copy that last read this buffer has finished
        cnt = min(_STAGE_BYTES, nbytes - off)
        bufs[b][:cnt].copy_(src[off:off + cnt])
        dst[off:off + cnt].copy_(bufs[b][:cnt], non_blocking=True)
        evs[b].record()
        k += 1
    evs[0].synchronize()
    evs[1].synchronize()
    return out


def _ptr(t):
    if t is None:
        return None
    assert t.is_cuda and t.dtype in (torch.float64, torch.int32, torch.int64, torch.uint8), (t.dtype, t.device)
    assert t.is_contiguous()
    return C.c_void_p(t.data_ptr())


def vec(t, per_chain_elems=None) -> Vec:
    """Build an omc_vec_t.  `t` is None (default), a shared tensor (stride 0) or a per-chain tensor [C, ...]."""
    if t is None:
        return Vec(None, 0)
    if isinstance(t, tuple):  # (tensor, explicit stride in elements)
        return Vec(t[0].data_ptr(), int(t[1]))
    if per_chain_elems is None:
        return Vec(t.data_ptr(), 0)
    return Vec(t.data_ptr(), int(per_chain_elems))


def rng(seed=0, sweep=None, chain_offset=0, site=0) -> Rng:
    if not 0 <= int(site) < 4096:
        raise ValueError(f"rng site {site}: the Philox counter gives a site 12 bits (4096 samplers per plan)")
    return Rng(int(seed) & 0xFFFFFFFFFFFFFFFF, sweep.data_ptr() if sweep is not None else None, int(chain_offset),
               int(site))


def counter_add(counter, inc=1):
    check(lib().omc_counter_add(_ptr(counter), int(inc), stream_ptr()), "omc_counter_add")


def counter_add2(c0, inc0, c1, inc1):
    check(lib().omc_counter_add2(_ptr(c0), int(inc0), _ptr(c1), int(inc1), stream_ptr()), "omc_counter_add2")


# ----------------------------------------------------------------------------- conjugate regression
def reg_pass_workspace(n_chains, n, p):
    ns = C.c_int(0)
    ws = C.c_longlong(0)
    check(lib().omc_reg_pass_workspace(n_chains, n, p, C.byref(ns), C.byref(ws)), "omc_reg_pass_workspace")
    return ns.value, ws.value


def reg_pass(X, y, w, beta, stats, workspace, n_chains, n, p, x_shared=False, y_shared=False, w_shared=False):
    """stats[c] = [X'WX | X'Wy | rss | cnt] for every chain (one fused pass over X)."""
    check(
        lib().omc_reg_pass(
            _ptr(X), 0 if x_shared else n * p, _ptr(y), 0 if y_shared else n, _ptr(w), 0 if w_shared else n,
            _ptr(beta), p, n_chains, n, p, _ptr(stats), _ptr(workspace), stream_ptr()),
        "omc_reg_pass",
    )


def reg_rss(X, y, w, beta, stats, workspace, n_chains, n, p, x_shared=False, y_shared=False, w_shared=False):
    """Residual-only pass: stats[c][rss | cnt] for the current beta; the G | g part of the record is left untouched."""
    check(
        lib().omc_reg_rss(
            _ptr(X), 0 if x_shared else n * p, _ptr(y), 0 if y_shared else n, _ptr(w), 0 if w_shared else n,
            _ptr(beta), p, n_chains, n, p, _ptr(stats), _ptr(workspace), stream_ptr()),
        "omc_reg_rss",
    )


def nn_dense_workspace(n_chains, p) -> int:
    """Doubles of scratch omc_nn_dense_draw / omc_dense_factor need (0 while the matrix fits in shared memory)."""
    d = C.c_longlong(0)
    check(lib().omc_nn_dense_workspace(int(n_chains), int(p), C.byref(d)), "omc_nn_dense_workspace")
    return d.value


def nn_dense_draw(n_chains, p, stats, tau, prior_kind, prior_P, lam, mu0, beta, rng_, debug_z=None, probe_Q=None,
                  probe_b=None, probe_L=None, probe_mu=None, status=None, debug_sweep_stride=0, trunc=None,
                  debug_u=None, center=None, rss_out=None, solve_only=False, ridge_rel=0.0, workspace=None):
    """trunc = (lo_vec, lo_len, hi_vec, hi_len) switches to the truncated-prior Gibbs scan (omc.h).
    center [C, 2p+1] (beta_hat | c0 | rss0) + rss_out (pointer into the record's rss slot): the draw also leaves
    rss(beta) there (re-centred sufficient statistics); solve_only: beta = posterior mean of the jittered system."""
    a = _cabi.NNDense()
    if trunc is not None:
        a.truncated = 1
        a.trunc_lo, a.trunc_lo_len, a.trunc_hi, a.trunc_hi_len = trunc
        a.debug_u = debug_u.data_ptr() if debug_u is not None else None
    a.n_chains, a.p = n_chains, p
    a.stats = Vec(stats.data_ptr(), p * p + p + 2)
    a.tau, a.prior_kind, a.prior_P, a.lam, a.mu0 = tau, prior_kind, prior_P, lam, mu0
    a.beta = beta.data_ptr()
    a.rng = rng_
    a.debug_z = debug_z.data_ptr() if debug_z is not None else None
    a.debug_sweep_stride = int(debug_sweep_stride)
    a.probe_Q = probe_Q.data_ptr() if probe_Q is not None else None
    a.probe_b = probe_b.data_ptr() if probe_b is not None else None
    a.probe_L = probe_L.data_ptr() if probe_L is not None else None
    a.probe_mu = probe_mu.data_ptr() if probe_mu is not None else None
    a.status = status.data_ptr() if status is not None else None
    if center is not None:
        a.center = Vec(center.data_ptr(), center.shape[1])
        a.rss_out = rss_out
    a.mode, a.ridge_rel = int(bool(solve_only)), float(ridge_rel)
    a.workspace = workspace.data_ptr() if workspace is not None else None
    check(lib().omc_nn_dense_draw(C.byref(a), stream_ptr()), "omc_nn_dense_draw")


EIGEN_MAX_P = 64


def eigen_record_len(p) -> int:
    """Doubles per chain of the eigen record M | D | h | m | u_hat | k (omc_nn_eigen_prep)."""
    return p * p + 5 * p


def nn_eigen_prep(n_chains, p, stats, prior_kind, prior_P, mu0, center, eig):
    """omc_nn_eigen_prep: per-chain eigenbasis M'P0M = I, M'GM = D of the records' G (P0 eye or diagonal) and the
    vectors the draw needs, into eig [C, p*p + 5p]; center [C, 2p+1] (beta_hat | c0 | rss0) or None."""
    a = _cabi.NNEigenPrep()
    a.n_chains, a.p = int(n_chains), int(p)
    a.stats = Vec(stats.data_ptr(), p * p + p + 2)
    a.prior_kind, a.prior_P, a.mu0 = int(prior_kind), prior_P, mu0
    a.center = Vec(center.data_ptr(), center.shape[1]) if center is not None else Vec(None, 0)
    a.eig = eig.data_ptr()
    check(lib().omc_nn_eigen_prep(C.byref(a), stream_ptr()), "omc_nn_eigen_prep")


def nn_eigen_draw(n_chains, p, eig, tau, lam, beta, rng_, status=None, debug_z=None, debug_sweep_stride=0, center=None,
                  rss_out=None, rss_stride=0):
    """omc_nn_eigen_draw: beta = M u from the eigen record; with center and rss_out (a pointer, rss_stride doubles
    between chains) also rss(beta)."""
    a = _cabi.NNEigenDraw()
    a.n_chains, a.p = int(n_chains), int(p)
    a.eig = eig.data_ptr()
    a.tau, a.lam = tau, lam
    a.beta = beta.data_ptr()
    a.rng = rng_
    a.debug_z = debug_z.data_ptr() if debug_z is not None else None
    a.debug_sweep_stride = int(debug_sweep_stride)
    a.status = status.data_ptr() if status is not None else None
    if center is not None:
        a.center = Vec(center.data_ptr(), center.shape[1])
        a.rss_out, a.rss_stride = rss_out, int(rss_stride)
    check(lib().omc_nn_eigen_draw(C.byref(a), stream_ptr()), "omc_nn_eigen_draw")


def dense_factor(Q, n, b=None, z=None, L=None, logdet=None, mean=None, x=None, status=None, factored=False,
                 backward_only=False, workspace=None, n_mats=None):
    """omc_dense_factor: blocked Cholesky / solves of n_mats dense SPD matrices [n_mats, n, n] (omc.h)."""
    a = _cabi.DenseFactor()
    m = int(n_mats if n_mats is not None else (Q.shape[0] if Q.dim() == 3 else 1))
    a.n_mats, a.n = m, int(n)
    a.Q, a.Q_stride = Q.data_ptr(), (n * n if Q.dim() == 3 and Q.shape[0] == m else 0)
    for name, t in (("b", b), ("z", z), ("L", L), ("logdet", logdet), ("mean", mean), ("x", x), ("status", status),
                    ("workspace", workspace)):
        setattr(a, name, t.data_ptr() if t is not None else None)
    a.factored, a.backward_only = int(bool(factored)), int(backward_only)
    check(lib().omc_dense_factor(C.byref(a), stream_ptr()), "omc_dense_factor")


def _quadform_args(n_chains, p, x, mu, kind, P, ss, cnt):
    a = _cabi.Quadform()
    a.n_chains, a.p, a.x, a.mu, a.kind, a.P = n_chains, p, x, mu, kind, P
    a.ss, a.cnt = ss.data_ptr(), cnt.data_ptr()
    return a


def quadform(n_chains, p, x, mu, kind, P, ss, cnt):
    a = _quadform_args(n_chains, p, x, mu, kind, P, ss, cnt)
    check(lib().omc_quadform(C.byref(a), stream_ptr()), "omc_quadform")


def _ng_draw_args(n_chains, a0, b0, ss, cnt, out, rng_, debug_g=None, probe_a=None, probe_b=None, debug_sweep_stride=0,
                  n_elem=0, a0_len=1, b0_len=1, ss_stride=0, cnt_stride=0):
    """n_elem > 0: vector-valued update, element k reads ss[k*ss_stride], cnt[k*cnt_stride] (omc.h)."""
    a = _cabi.NGDraw()
    a.n_elem, a.a0_len, a.b0_len, a.ss_stride, a.cnt_stride = int(n_elem), int(a0_len), int(b0_len), int(ss_stride), int(cnt_stride)
    a.n_chains, a.a0, a.b0, a.ss, a.cnt = n_chains, a0, b0, ss, cnt
    a.out = out.data_ptr()
    a.rng = rng_
    a.debug_g = debug_g.data_ptr() if debug_g is not None else None
    a.debug_sweep_stride = int(debug_sweep_stride)
    a.probe_a = probe_a.data_ptr() if probe_a is not None else None
    a.probe_b = probe_b.data_ptr() if probe_b is not None else None
    return a


def ng_draw(*args, **kw):
    """Gamma(a0 + cnt / 2, b0 + ss / 2) draws (omc.h); n_elem > 0: vector-valued update."""
    a = _ng_draw_args(*args, **kw)
    check(lib().omc_ng_draw(C.byref(a), stream_ptr()), "omc_ng_draw")


# ----------------------------------------------------------------------------- mixture models (SURVEY f2)
def mixture_allocation(n_chains, n, K, x, mu, tau, prob, prob_rows, z, rng_, debug_u=None, debug_sweep_stride=0):
    a = _cabi.MixtureAlloc()
    a.n_chains, a.n, a.K, a.x, a.mu, a.tau, a.prob, a.prob_rows = n_chains, n, K, x, mu, tau, prob, int(prob_rows)
    a.z = z.data_ptr()
    a.rng = rng_
    a.debug_u = debug_u.data_ptr() if debug_u is not None else None
    a.debug_sweep_stride = int(debug_sweep_stride)
    check(lib().omc_mixture_allocation(C.byref(a), stream_ptr()), "omc_mixture_allocation")


def mixture_stats(n_chains, n, K, x, mu, tau, z, stats, record=None, gather_mu=None, gather_tau=None, logp=None,
                  accumulate=False):
    a = _cabi.MixtureStats()
    a.n_chains, a.n, a.K, a.x, a.mu, a.tau = n_chains, n, K, x, mu, tau
    a.z, a.stats = z.data_ptr(), stats.data_ptr()
    a.record, a.gather_mu, a.gather_tau, a.logp = _ptr(record), _ptr(gather_mu), _ptr(gather_tau), _ptr(logp)
    a.accumulate = int(bool(accumulate))
    check(lib().omc_mixture_stats(C.byref(a), stream_ptr()), "omc_mixture_stats")


def logp_categorical(n_chains, n, K, z, prob, prob_rows, out, accumulate):
    check(lib().omc_logp_categorical(n_chains, n, K, _ptr(z), prob, int(prob_rows), _ptr(out), int(bool(accumulate)),
                                     stream_ptr()), "omc_logp_categorical")


# ----------------------------------------------------------------------------- log densities / predictors
def logp_normal_ss(n_chains, dim, ss, scalar, logdet, out, accumulate):
    a = _cabi.LogpNormalSS(n_chains, float(dim), ss, scalar, logdet, out.data_ptr(), int(accumulate))
    check(lib().omc_logp_normal_ss(C.byref(a), stream_ptr()), "omc_logp_normal_ss")


def logp_gamma(n_chains, n_elem, x, shape, shape_len, rate, rate_len, out, accumulate):
    a = _cabi.LogpGamma(n_chains, n_elem, shape_len, rate_len, x, shape, rate, out.data_ptr(), int(accumulate))
    check(lib().omc_logp_gamma(C.byref(a), stream_ptr()), "omc_logp_gamma")


def logp_poisson(n_chains, n_elem, k, rate, rate_len, out, accumulate):
    a = _cabi.LogpPoisson(n_chains, n_elem, rate_len, k, rate, out.data_ptr(), int(accumulate))
    check(lib().omc_logp_poisson(C.byref(a), stream_ptr()), "omc_logp_poisson")


def logp_domain(n_chains, n_elem, x, lower, lo_len, upper, hi_len, out):
    check(lib().omc_logp_domain(n_chains, n_elem, x, lower, int(lo_len), upper, int(hi_len), _ptr(out), stream_ptr()),
          "omc_logp_domain")


def logp_const(value, n_chains, out, accumulate):
    check(lib().omc_logp_const(float(value), n_chains, _ptr(out), int(accumulate), stream_ptr()), "omc_logp_const")


def linear_predictor(n_chains, n, terms, out, residual_of=None):
    """terms: list of (X_vec, theta_vec, p[, transform_exp]); residual_of (omc_vec_t): out = residual_of - yhat."""
    a = _cabi.LinearPredictor()
    if residual_of is not None:
        a.residual_of = residual_of
    a.n_chains, a.n, a.n_terms = n_chains, n, len(terms)
    for i, (xv, tv, p, *rest) in enumerate(terms):
        a.p[i] = p
        a.X[i] = xv
        a.theta[i] = tv
        a.transform_exp[i] = int(bool(rest[0])) if rest else 0
    a.out = out.data_ptr()
    check(lib().omc_linear_predictor(C.byref(a), stream_ptr()), "omc_linear_predictor")


def combine(n_chains, length, xs, scales, out):
    """out[c][i] = sum_t scales[t][c] * xs[t][c][i]; xs / scales: lists of omc_vec_t (scale None => 1)."""
    n = len(xs)
    X = (Vec * n)(*xs)
    S = (Vec * n)(*[s if s is not None else Vec(None, 0) for s in scales])
    check(lib().omc_combine(int(n_chains), int(length), n, X, S, _ptr(out), stream_ptr()), "omc_combine")


def sum_log(x, n, out):
    check(lib().omc_sum_log(_ptr(x), out.numel(), int(n), _ptr(out), stream_ptr()), "omc_sum_log")


def log_elements(x, out):
    check(lib().omc_log_elements(_ptr(x), x.numel(), _ptr(out), stream_ptr()), "omc_log_elements")


def logdet_dense(P, n, out):
    """log|P| of out.numel() dense SPD matrices; above n = 64 through the blocked factorisation (omc_dense_factor)."""
    if n <= 64:
        check(lib().omc_logdet_dense(_ptr(P), out.numel(), int(n), _ptr(out), stream_ptr()), "omc_logdet_dense")
        return
    m = out.numel()
    ws = nn_dense_workspace(m, n)
    work = torch.empty(ws, dtype=torch.float64, device=P.device) if ws else None
    dense_factor(P.reshape(m, n, n), n, logdet=out, workspace=work, n_mats=m)


# ----------------------------------------------------------------------------- fused per-chain small ops
FUSED_COPY_MAX = 4 << 20     # store copies above this many doubles keep their own (wider) kernel


def _fop(kind, field, value):
    f = _cabi.FOp()
    f.kind = kind
    setattr(f.u, field, value)
    return f


def fop_logp_normal_ss(n_chains, dim, ss, scalar, logdet, out, accumulate):
    return _fop(_cabi.FOP_LOGP_NORMAL_SS, "normal_ss",
                _cabi.LogpNormalSS(n_chains, float(dim), ss, scalar, logdet, out.data_ptr(), int(accumulate)))


def fop_logp_gamma(n_chains, n_elem, x, shape, shape_len, rate, rate_len, out, accumulate):
    return _fop(_cabi.FOP_LOGP_GAMMA, "gamma",
                _cabi.LogpGamma(n_chains, n_elem, shape_len, rate_len, x, shape, rate, out.data_ptr(), int(accumulate)))


def fop_logp_poisson(n_chains, n_elem, k, rate, rate_len, out, accumulate):
    return _fop(_cabi.FOP_LOGP_POISSON, "poisson",
                _cabi.LogpPoisson(n_chains, n_elem, rate_len, k, rate, out.data_ptr(), int(accumulate)))


def fop_logp_const(value, n_chains, out, accumulate):
    return _fop(_cabi.FOP_LOGP_CONST, "konst", _cabi._FKonst(float(value), out.data_ptr(), int(accumulate)))


def fop_ng_draw(*args, **kw):
    return _fop(_cabi.FOP_NG_DRAW, "ng", _ng_draw_args(*args, **kw))


def fop_quadform(n_chains, p, x, mu, kind, P, ss, cnt):
    return _fop(_cabi.FOP_QUADFORM, "quad", _quadform_args(n_chains, p, x, mu, kind, P, ss, cnt))


def fop_store_copy(src, dst, count, iter_counter, max_iter, ring=False):
    return _fop(_cabi.FOP_STORE_COPY, "copy", _cabi._FCopy(src.data_ptr(), dst.data_ptr(), int(count), iter_counter.data_ptr(),
                                                          int(max_iter), int(bool(ring))))


def fused_small(n_chains, fops):
    """One launch running `fops` (omc_fop_t descriptors) in order; returns the launch closure (owns the argument block)."""
    a = _cabi.FusedSmall()
    a.n_chains, a.n_ops = int(n_chains), len(fops)
    for i, f in enumerate(fops):
        a.ops[i] = f

    def launch():
        check(lib().omc_fused_small(C.byref(a), stream_ptr()), "omc_fused_small")

    return launch


# ----------------------------------------------------------------------------- graphs / schedule
class Graph:
    """A captured CUDA graph of op launches (omc_graph_t)."""

    def __init__(self, handle):
        self.handle = handle

    @staticmethod
    def capture(fn):
        """Record every libomc launch `fn()` makes on the current stream into a replayable graph."""
        st = stream_ptr()
        check(lib().omc_graph_capture_begin(st), "omc_graph_capture_begin")
        try:
            fn()
        finally:
            h = C.c_void_p()
            rc = lib().omc_graph_capture_end(st, C.byref(h))
        check(rc, "omc_graph_capture_end")
        return Graph(h)

    def launch(self, times=1):
        check(lib().omc_graph_launch(self.handle, stream_ptr(), int(times)), "omc_graph_launch")

    def num_kernels(self) -> int:
        n = C.c_longlong(0)
        check(lib().omc_graph_num_kernel_nodes(self.handle, C.byref(n)), "omc_graph_num_kernel_nodes")
        return n.value

    def __del__(self):
        try:
            if self.handle:
                lib().omc_graph_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


def run_schedule(sweep: Graph, store, n_burn, n_iter, n_thin):
    check(
        lib().omc_run_schedule(sweep.handle, store.handle if store is not None else None, stream_ptr(), int(n_burn),
                               int(n_iter), int(n_thin)),
        "omc_run_schedule",
    )


def store_copy(src, dst, count, iter_counter, max_iter, ring=False):
    """Row *iter_counter of a [max_iter, count] store, or (ring=True) slab *iter_counter % max_iter of a ring."""
    fn = lib().omc_store_copy_ring if ring else lib().omc_store_copy
    check(fn(_ptr(src), _ptr(dst), int(count), _ptr(iter_counter), int(max_iter), stream_ptr()), "omc_store_copy")


# ----------------------------------------------------------------------------- Metropolis-Hastings family
TERM_POISSON_RATE, TERM_GAMMA_RESPONSE, TERM_NORMAL_RESPONSE, TERM_UNIFORM_RESPONSE = 1, 2, 3, 4
TERM_LOGNORMAL_RESPONSE, TERM_NORMAL_LINEAR = 5, 6


def term(kind, mat_kind=0, p1_len=1, p2_len=1, data=None, p1=None, p2=None, P=None, scalar=None, logdet=None,
         dom_lo=float("-inf"), dom_hi=float("inf"), stats=None, n_data=0, transform_exp=False) -> "_cabi.Term":
    """Build an omc_term_t; operands are omc_vec_t (see `vec`) or None."""
    none = Vec(None, 0)
    return _cabi.Term(int(kind), int(mat_kind), int(p1_len), int(p2_len), data or none, p1 or none, p2 or none,
                      P or none, scalar or none, logdet or none, float(dom_lo), float(dom_hi), stats or none,
                      int(n_data), int(bool(transform_exp)))


def mh_model(n_chains, n_elem, terms) -> "_cabi.MHModel":
    if len(terms) > 4:
        raise _cabi.OmcError("the device MH model supports at most 4 terms in the conditional model")
    m = _cabi.MHModel()
    m.n_chains, m.n_elem, m.n_terms = int(n_chains), int(n_elem), len(terms)
    for i, t in enumerate(terms):
        m.terms[i] = t
    return m


def mh_logp(model, theta, out, accumulate=False):
    check(lib().omc_mh_logp_acc(C.byref(model), _ptr(theta), _ptr(out), int(bool(accumulate)), stream_ptr()),
          "omc_mh_logp")


def mh_grad_hess(model, theta, method, grad, hess=None):
    """method: 0 analytic, 1 the reference's finite-difference stencil.  hess must be zero-initialised by the kernel."""
    check(lib().omc_mh_grad_hess(C.byref(model), _ptr(theta), int(method), _ptr(grad), _ptr(hess), stream_ptr()),
          "omc_mh_grad_hess")


def random_walk(model, theta, p_dim, n_rep, loop, step, step_rows, step_cols, limits, rng_, debug_z=None, debug_u=None,
                stride_z=0, stride_u=0, counters=None, probe=None):
    a = _cabi.RandomWalkArgs()
    a.model = model
    a.theta = theta.data_ptr()
    a.p_dim, a.n_rep, a.loop = int(p_dim), int(n_rep), int(loop)
    a.step, a.step_rows, a.step_cols = step, int(step_rows), int(step_cols)
    a.limits = limits.data_ptr() if limits is not None else None
    a.rng = rng_
    a.debug_z = debug_z.data_ptr() if debug_z is not None else None
    a.debug_u = debug_u.data_ptr() if debug_u is not None else None
    a.debug_sweep_stride_z, a.debug_sweep_stride_u = int(stride_z), int(stride_u)
    a.counters = counters.data_ptr() if counters is not None else None
    a.probe = probe.data_ptr() if probe is not None else None
    check(lib().omc_random_walk(C.byref(a), stream_ptr()), "omc_random_walk")


def mmala(model, theta, step, method, rng_, debug_z=None, debug_u=None, stride_z=0, stride_u=0, counters=None,
          status=None, probe_mu=None, probe_L=None, probe_prop=None, probe_scalars=None, workspace=None):
    """workspace: nn_dense_workspace(n_chains, n_elem) doubles when that is > 0 (dense Hessian above n_elem = 136)."""
    a = _cabi.MMalaArgs()
    a.model = model
    a.theta = theta.data_ptr()
    a.step, a.method = float(step), int(method)
    a.rng = rng_
    a.debug_z = debug_z.data_ptr() if debug_z is not None else None
    a.debug_u = debug_u.data_ptr() if debug_u is not None else None
    a.debug_sweep_stride_z, a.debug_sweep_stride_u = int(stride_z), int(stride_u)
    for name, t in (("counters", counters), ("status", status), ("probe_mu", probe_mu), ("probe_L", probe_L),
                    ("probe_prop", probe_prop), ("probe_scalars", probe_scalars), ("workspace", workspace)):
        setattr(a, name, t.data_ptr() if t is not None else None)
    check(lib().omc_mmala(C.byref(a), stream_ptr()), "omc_mmala")


def truncnorm_rv(mean, scale, lower, upper, u, out):
    check(lib().omc_truncnorm_rv(_ptr(mean), _ptr(scale), _ptr(lower), _ptr(upper), _ptr(u), out.numel(), _ptr(out),
                                 stream_ptr()), "omc_truncnorm_rv")


def truncnorm_logpdf(x, mean, scale, lower, upper, out):
    check(lib().omc_truncnorm_logpdf(_ptr(x), _ptr(mean), _ptr(scale), _ptr(lower), _ptr(upper), out.numel(),
                                     _ptr(out), stream_ptr()), "omc_truncnorm_logpdf")


# ----------------------------------------------------------------------------- temporal GMRF (tridiagonal precision)
def tridiag_workspace(n_chains, n) -> int:
    b = C.c_longlong(0)
    check(lib().omc_tridiag_workspace(int(n_chains), int(n), C.byref(b)), "omc_tridiag_workspace")
    return b.value


def tridiag_args(n_chains, n, pd, pe, workspace, lam=None, tau=None, w=None, y=None, h=None, mu0=None, x=None,
                 rng_=None, debug_z=None, debug_sweep_stride=0, ss_prior=None, ss_lik=None, logdet=None, probe_l=None,
                 probe_c=None, status=None) -> "_cabi.TridiagNN":
    """Build an omc_tridiag_nn_t.  lam/tau/w/y/h/mu0 are omc_vec_t (see `vec`) or None; the rest tensors or None."""
    none = Vec(None, 0)
    a = _cabi.TridiagNN()
    a.n_chains, a.n = int(n_chains), int(n)
    a.pd, a.pe = pd.data_ptr(), (pe.data_ptr() if pe is not None and pe.numel() else None)
    a.lam, a.tau, a.w, a.y, a.h, a.mu0 = lam or none, tau or none, w or none, y or none, h or none, mu0 or none
    a.x = x.data_ptr() if x is not None else None
    a.rng = rng_ if rng_ is not None else Rng(0, None, 0, 0)
    a.debug_z = debug_z.data_ptr() if debug_z is not None else None
    a.debug_sweep_stride = int(debug_sweep_stride)
    for name, t in (("ss_prior", ss_prior), ("ss_lik", ss_lik), ("logdet", logdet), ("probe_l", probe_l),
                    ("probe_c", probe_c), ("status", status)):
        setattr(a, name, t.data_ptr() if t is not None else None)
    a.workspace = workspace.data_ptr()
    return a


def tridiag_nn_draw(args):
    check(lib().omc_tridiag_nn_draw(C.byref(args), stream_ptr()), "omc_tridiag_nn_draw")


def tridiag_quadforms(args):
    check(lib().omc_tridiag_quadforms(C.byref(args), stream_ptr()), "omc_tridiag_quadforms")


def bidiag_gram(l, c, n, pd, pe):
    """pd, pe <- diagonals of L L' for a lower bidiagonal L (diagonal l, sub-diagonal c)."""
    check(lib().omc_bidiag_gram(_ptr(l), _ptr(c) if c is not None and c.numel() else None, int(n), _ptr(pd),
                                _ptr(pe) if pe is not None and pe.numel() else None, stream_ptr()), "omc_bidiag_gram")


def tridiag_matvec(pd, pe, v, n_chains, n, out):
    check(lib().omc_tridiag_matvec(_ptr(pd), _ptr(pe) if pe is not None and pe.numel() else None, v, int(n_chains),
                                   int(n), _ptr(out), stream_ptr()), "omc_tridiag_matvec")


# ----------------------------------------------------------------------------- ReversibleJump (Gaussian-kernel basis)
def rj_args(n_chains, n_data, n_max, n_basis, theta, omega, beta, B, X, theta_lo, theta_hi, birth_probability=0.5,
            y=None, tau_y=None, sample_omega=True, omega_shape=None, omega_rate=None, mu_beta=None, tau_beta=None,
            rho=None, match_scale=1.0, match_limits=None, rng_=None, debug=None, debug_sweep_stride=0, counters=None,
            status=None, probe=None, logp_out=None, size_class=None, gram=None, gram_valid=None) -> "_cabi.RJArgs":
    """Build an omc_rj_t.  State tensors are padded to n_max; y/tau_y/... are omc_vec_t (see `vec`) or None."""
    none = Vec(None, 0)
    a = _cabi.RJArgs()
    a.n_chains, a.n_data, a.n_max = int(n_chains), int(n_data), int(n_max)
    a.n_basis, a.theta, a.omega, a.beta, a.B, a.X = (t.data_ptr() for t in (n_basis, theta, omega, beta, B, X))
    a.y, a.tau_y = y or none, tau_y or none
    a.theta_lo, a.theta_hi = float(theta_lo), float(theta_hi)
    a.sample_omega = int(bool(sample_omega))
    a.omega_shape, a.omega_rate = omega_shape or none, omega_rate or none
    a.mu_beta, a.tau_beta, a.rho = mu_beta or none, tau_beta or none, rho or none
    a.birth_probability, a.match_scale = float(birth_probability), float(match_scale)
    a.match_truncated = int(match_limits is not None)
    a.match_lo, a.match_hi = (float(match_limits[0]), float(match_limits[1])) if match_limits is not None else (0.0, 0.0)
    a.rng = rng_ if rng_ is not None else Rng(0, None, 0, 0)
    a.debug = debug.data_ptr() if debug is not None else None
    a.debug_sweep_stride = int(debug_sweep_stride)
    for name, t in (("counters", counters), ("status", status), ("probe", probe), ("logp_out", logp_out),
                    ("size_class", size_class), ("gram", gram), ("gram_valid", gram_valid)):
        setattr(a, name, t.data_ptr() if t is not None else None)
    a.logp_only = 0
    return a


def reversible_jump(args, logp_only=False):
    args.logp_only = int(logp_only)
    check(lib().omc_reversible_jump(C.byref(args), stream_ptr()), "omc_reversible_jump")
    args.logp_only = 0


def rj_basis(args):
    check(lib().omc_rj_basis(C.byref(args), stream_ptr()), "omc_rj_basis")


def rj_knot_walk(rj_args_, which, step, lim_lo, lim_hi, debug_tn_u=None, debug_u=None, debug_sweep_stride=0,
                 counters=None, rng_=None):
    """RandomWalkLoop over the knots (which = 0) / widths (which = 1) of the padded RJ state (omc.h)."""
    w = _cabi.RJWalk()
    C.memmove(C.byref(w.model), C.byref(rj_args_), C.sizeof(_cabi.RJArgs))
    if rng_ is not None:
        w.model.rng = rng_
    w.which, w.step, w.lim_lo, w.lim_hi = int(which), float(step), float(lim_lo), float(lim_hi)
    w.debug_tn_u = debug_tn_u.data_ptr() if debug_tn_u is not None else None
    w.debug_u = debug_u.data_ptr() if debug_u is not None else None
    w.debug_sweep_stride = int(debug_sweep_stride)
    w.counters = counters.data_ptr() if counters is not None else None
    check(lib().omc_rj_knot_walk(C.byref(w), stream_ptr()), "omc_rj_knot_walk")


def rj_coef_mmala(rj_args_, step, debug_z=None, debug_u=None, stride_z=0, stride_u=0, counters=None, probe=None,
                  rng_=None):
    """ManifoldMALA on the live coefficients of the padded RJ state (omc.h)."""
    m = _cabi.RJMmala()
    C.memmove(C.byref(m.model), C.byref(rj_args_), C.sizeof(_cabi.RJArgs))
    if rng_ is not None:
        m.model.rng = rng_
    m.step = float(step)
    m.debug_z = debug_z.data_ptr() if debug_z is not None else None
    m.debug_u = debug_u.data_ptr() if debug_u is not None else None
    m.debug_sweep_stride_z, m.debug_sweep_stride_u = int(stride_z), int(stride_u)
    m.counters = counters.data_ptr() if counters is not None else None
    m.probe = probe.data_ptr() if probe is not None else None
    check(lib().omc_rj_coef_mmala(C.byref(m), stream_ptr()), "omc_rj_coef_mmala")
