"""GPU: the log-density, predictor and store-epilogue kernels (logp.cu, fused_small.cu, omc_api.cu), each called through
its kernels.py wrapper and compared with what the reference's own call returns: scipy.stats per element summed per chain
with math.fsum, the formula of oracle/dist.normal_log_p_from_ss, numpy.linalg.slogdet, plain fp64 numpy.

Where these kernels go wrong is covered on purpose: the 256-element block stride of logp.cu, the 32-lane stride of
fused_small.cu and its switch from one lane to 32 lanes per chain above 4 elements, parameters broadcast (length 1) or
per element, shared operands (chain stride 0), accumulate, and scipy's support and invalid-parameter conventions.

Tolerance: a finite result r of a sum satisfies |r - ref| <= 8 eps M, where M sums the magnitudes of every addend of
the reference formula (for the Gamma: |xlogy(a-1, y)| + |y| + |gammaln(a)| + |log scale| per element) -- the scale a
double evaluation of that formula is accurate to, whatever the order of the sum and however much the total cancels.
A non-finite result must have the reference's class exactly (NaN, +inf or -inf).
ref: distribution.py:241-261 (Gamma), 490-508 (Poisson), location_scale.py:145-167, mcmc.py:105-111 (store epilogue).
"""

import math

import numpy as np
import pytest
from scipy import special, stats

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps
NAN, INF = float("nan"), float("inf")
NS = (0, 1, 4, 5, 31, 32, 33, 255, 256, 257, 1000, 4099)
# logp_cu: the stand-alone kernel; fused: one fused_small op alone (one lane per chain up to 4 elements, a warp above);
# fused_warp: the same op next to a 40-element quadratic form, which makes the launch run 32 lanes per chain
IMPLS = ("logp_cu", "fused", "fused_warp")


@pytest.fixture(autouse=True, scope="module")
def _device():
    from openmcmc_b200 import kernels as K

    K.init_device(0)


def _t(a):
    import torch

    return torch.tensor(np.ascontiguousarray(a, dtype=np.float64), device="cuda")


def _host(t):
    import torch

    torch.cuda.synchronize()
    return t.cpu().numpy()


def _fsum(terms):
    """math.fsum with IEEE classes: NaN if a term is NaN or +inf meets -inf, else the infinity, else the exact sum."""
    terms = np.asarray(terms, dtype=np.float64).ravel()
    if np.isnan(terms).any() or ((terms == INF).any() and (terms == -INF).any()):
        return NAN
    if np.isinf(terms).any():
        return terms[np.isinf(terms)][0]
    return math.fsum(terms)


def _check(got, ref, mag, what):
    """Element-wise: the reference's class where it is not finite, |got - ref| <= 8 eps mag where it is."""
    ref = np.asarray(ref, dtype=np.float64)
    mag = np.broadcast_to(np.asarray(mag, dtype=np.float64), ref.shape).ravel()
    got, ref = np.asarray(got, dtype=np.float64).ravel(), ref.ravel()
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    nan, inf = np.isnan(ref), np.isinf(ref)
    fin = ~(nan | inf)
    ok = np.empty(ref.shape, dtype=bool)
    ok[nan] = np.isnan(got[nan])
    ok[inf] = got[inf] == ref[inf]
    with np.errstate(invalid="ignore"):
        ok[fin] = np.isfinite(got[fin]) & (np.abs(got[fin] - ref[fin]) <= 8 * EPS * mag[fin])
    if not ok.all():
        i = np.flatnonzero(~ok)[0]
        raise AssertionError(f"{what}: {np.count_nonzero(~ok)} of {ref.size} wrong, first [{i}]: got {got[i]!r}, "
                             f"expected {ref[i]!r} (tolerance {8 * EPS * mag[i]:.3g})")


# ----------------------------------------------------------------------------- scipy per element
def _gamma_terms(x, shape, rate):
    """stats.gamma.logpdf(x, a, scale=1/rate) per element and the magnitude of its addends."""
    with np.errstate(all="ignore"):
        scale = 1.0 / np.asarray(rate, dtype=np.float64)
        lp = stats.gamma.logpdf(x, shape, scale=scale)
        y = x / scale
        mag = np.abs(special.xlogy(shape - 1.0, y)) + np.abs(y) + np.abs(special.gammaln(shape)) + np.abs(np.log(scale))
    return lp, mag


def _poisson_terms(k, mu):
    """stats.poisson.logpmf(k, mu) per element and the magnitude of its addends."""
    with np.errstate(all="ignore"):
        lp = stats.poisson.logpmf(k, mu)
        mag = np.abs(special.xlogy(k, mu)) + np.abs(special.gammaln(k + 1.0)) + np.abs(mu)
    return lp, mag


def _chain_sums(lp, mag):
    """Per chain (rows): the fsum of the log-densities and the sum of the magnitudes where the sum is finite."""
    ref = np.array([_fsum(r) for r in lp]) if lp.shape[1] else np.zeros(lp.shape[0])
    m = np.array([math.fsum(r[np.isfinite(r)]) for r in mag]) if lp.shape[1] else np.zeros(lp.shape[0])
    return ref, m


# ----------------------------------------------------------------------------- launching one op three ways
class _Ops:
    """Keeps every tensor an omc_vec_t points at alive until the launch has finished."""

    def __init__(self, C):
        self.C, self.keep = C, []

    def dev(self, a):
        t = _t(a)
        self.keep.append(t)
        return t

    def param(self, full, length, shared):
        """Device operand of a parameter: length 1 or n_elem, per chain or shared (stride 0).  `full` is [C, length]."""
        from openmcmc_b200 import kernels as K

        if shared:
            return K.vec(self.dev(full[0, :length]))
        return K.vec(self.dev(full[:, :length]), length)

    def lane_forcer(self):
        """A 40-element quadratic form: the widest op of the launch then has more than 4 elements (32 lanes per chain)."""
        from openmcmc_b200 import kernels as K

        x = self.dev(np.ones((self.C, 40)))
        ss, cnt = self.dev(np.zeros(self.C)), self.dev(np.zeros(self.C))
        return K.fop_quadform(self.C, 40, K.vec(x, 40), K.vec(None), K.MAT_EYE, K.vec(None), ss, cnt)

    def run(self, impl, standalone, fop):
        from openmcmc_b200 import kernels as K

        if impl == "logp_cu":
            standalone()
        else:
            K.fused_small(self.C, [fop] + ([self.lane_forcer()] if impl == "fused_warp" else []))()


def _run_gamma(ops, impl, n, x, sh, sh_len, rt, rt_len, out, acc):
    from openmcmc_b200 import kernels as K

    args = (ops.C, n, K.vec(ops.dev(x), n), sh, sh_len, rt, rt_len, out, acc)
    ops.run(impl, lambda: K.logp_gamma(*args), K.fop_logp_gamma(*args))


def _run_poisson(ops, impl, n, k, rt, rt_len, out, acc):
    from openmcmc_b200 import kernels as K

    args = (ops.C, n, K.vec(ops.dev(k), n), rt, rt_len, out, acc)
    ops.run(impl, lambda: K.logp_poisson(*args), K.fop_logp_poisson(*args))


def _param_lens(n):
    return sorted({1, max(n, 1)})


# ----------------------------------------------------------------------------- 1. Gamma / Poisson sums
def _random_case(dist, n, C):
    rng = np.random.default_rng(1000 * n + C + (0 if dist == "gamma" else 7))
    w = max(n, 1)
    if dist == "gamma":
        p1 = rng.uniform(0.3, 6.0, (C, w))                    # shape
        p2 = rng.uniform(0.2, 4.0, (C, w))                    # rate
        x = rng.gamma(2.0, 1.5, (C, n))
    else:
        p1 = None
        p2 = rng.uniform(0.05, 30.0, (C, w))                  # mean
        x = rng.poisson(rng.uniform(0.05, 30.0, (C, n))).astype(np.float64)
    return x, p1, p2


def _sums(dist, x, p1, p2, lens, shared):
    """Reference sums per chain for parameters of these lengths, per chain or taken from chain 0 (shared)."""
    C, n = x.shape

    def full(p, length):
        src = p[:1] if shared else p
        return np.broadcast_to(src[:, :length], (C, n)) if n else np.zeros((C, 0))

    if dist == "gamma":
        return _chain_sums(*_gamma_terms(x, full(p1, lens[0]), full(p2, lens[1])))
    return _chain_sums(*_poisson_terms(x, full(p2, lens[1])))


@pytest.mark.parametrize("dist,n,impl", [(d, n, i) for d in ("gamma", "poisson") for n in NS for i in IMPLS])
def test_logp_sum_against_scipy(dist, n, impl):
    """Random valid inputs at every boundary size, both parameter lengths, per-chain and shared parameters; accumulate = 0
    overwrites a NaN, accumulate = 1 adds to what `out` held."""
    import torch

    for C in (1, 7, 300):
        x, p1, p2 = _random_case(dist, n, C)
        prefill = np.random.default_rng(C).normal(0.0, 50.0, C)
        for lens in ([(a, b) for a in _param_lens(n) for b in _param_lens(n)] if dist == "gamma"
                     else [(1, b) for b in _param_lens(n)]):
            for shared in (False, True):
                ref, mag = _sums(dist, x, p1, p2, lens, shared)
                for acc in (0, 1):
                    ops = _Ops(C)
                    out = _t(prefill) if acc else torch.full((C,), NAN, dtype=torch.float64, device="cuda")
                    rt = ops.param(p2, lens[1], shared)
                    if dist == "gamma":
                        _run_gamma(ops, impl, n, x, ops.param(p1, lens[0], shared), lens[0], rt, lens[1], out, acc)
                    else:
                        _run_poisson(ops, impl, n, x, rt, lens[1], out, acc)
                    want = ref + (prefill if acc else 0.0)
                    _check(_host(out), want, mag + (np.abs(prefill) if acc else 0.0),
                           f"{dist} {impl} n={n} C={C} lens={lens} shared={shared} acc={acc}")


@pytest.mark.parametrize("dist,impl", [(d, i) for d in ("gamma", "poisson") for i in IMPLS])
def test_logp_one_hot_index(dist, impl):
    """Every element at a point of log-density exactly 0 (Poisson k = mu = 0; Gamma x = 0, shape = rate = 1) but one, at
    index 0, 31, 32, 255, 256 or n-1: the chain's sum is that one element's log-density, for every parameter layout."""
    import torch

    C = 7
    for n in NS[1:]:
        for i in sorted({j for j in (0, 31, 32, 255, 256) if j < n} | {n - 1}):
            for lens in ([(a, b) for a in _param_lens(n) for b in _param_lens(n)] if dist == "gamma"
                         else [(1, b) for b in _param_lens(n)]):
                for shared in (False, True):
                    ops = _Ops(C)
                    x = np.zeros((C, n))
                    x[:, i] = (1.5 + 0.75 * np.arange(C)) if dist == "gamma" else 1.0 + np.arange(C)   # one per chain
                    p1, p2 = np.ones((C, n)), (np.ones((C, n)) if dist == "gamma" else np.zeros((C, n)))
                    for L, p, base in ((lens[0], p1, 3.5), (lens[1], p2, 0.6 if dist == "gamma" else 2.5)):
                        if L > 1:                                   # per element: distinct at index i only
                            p[:, i] = base + 0.25 * np.arange(C)
                    if shared:
                        p1[:], p2[:] = p1[0], p2[0]
                    out = torch.full((C,), NAN, dtype=torch.float64, device="cuda")
                    rt = ops.param(p2, lens[1], shared)
                    if dist == "gamma":
                        _run_gamma(ops, impl, n, x, ops.param(p1, lens[0], shared), lens[0], rt, lens[1], out, 0)
                        ref, mag = _gamma_terms(x[:, i], p1[:, i], p2[:, i])
                    else:
                        _run_poisson(ops, impl, n, x, rt, lens[1], out, 0)
                        ref, mag = _poisson_terms(x[:, i], p2[:, i])
                    _check(_host(out), ref, mag, f"{dist} {impl} n={n} one-hot at {i} lens={lens} shared={shared}")


GAMMA_EDGES = [  # (x, shape, rate)
    (0.0, 0.5, 1.0), (0.0, 1.0, 1.0), (0.0, 2.5, 1.0),          # x = 0 with shape < 1, = 1, > 1: +inf, log rate, -inf
    (-1.0, 2.0, 1.0), (NAN, 2.0, 1.0), (INF, 2.0, 1.0), (INF, 1.0, 1.0), (INF, 0.5, 1.0),
    (1e-300, 2.0, 1.0), (1e300, 2.0, 1.0), (1e-300, 0.5, 1.3), (1e300, 0.5, 1.3),
    (1.0, 2.0, 0.0), (1.0, 1.0, 0.0), (1.0, 0.5, 0.0), (0.0, 0.5, 0.0), (-1.0, 2.0, 0.0),   # rate 0: scale = inf
    (1.0, 2.0, -1.0), (0.0, 2.0, -1.0), (-1.0, 2.0, -1.0),     # rate < 0: NaN
    (1.0, 0.0, 1.0), (-1.0, 0.0, 1.0), (1.0, -0.5, 1.0), (1.0, -2.0, 1.0), (NAN, -2.0, 1.0),   # shape <= 0: NaN
]
POISSON_EDGES = [  # (k, mu)
    (0.0, 0.0), (3.0, 0.0), (2.5, 1.0), (-1.0, 1.0), (NAN, 1.0), (1e6, 1e6),
    (0.0, -1.0), (2.0, -1.0), (2.5, -1.0), (-1.0, -1.0),           # mu < 0: NaN, whatever k
    (0.0, INF), (2.0, INF), (INF, 1.0), (0.0, NAN),
]


@pytest.mark.parametrize("dist,impl", [(d, i) for d in ("gamma", "poisson") for i in IMPLS])
def test_logp_edge_values(dist, impl):
    """One edge value per chain, among elements of log-density 0, at 4 elements (one lane per chain when fused alone)
    and 40: the class or the value scipy gives."""
    import torch

    edges = GAMMA_EDGES if dist == "gamma" else POISSON_EDGES
    C = len(edges)
    for n in (4, 40):
        ops = _Ops(C)
        x, p1, p2 = np.zeros((C, n)), np.ones((C, n)), (np.ones((C, n)) if dist == "gamma" else np.zeros((C, n)))
        at = [(7 * c) % n for c in range(C)]
        for c, e in enumerate(edges):
            if dist == "gamma":
                x[c, at[c]], p1[c, at[c]], p2[c, at[c]] = e
            else:
                x[c, at[c]], p2[c, at[c]] = e
        out = torch.full((C,), NAN, dtype=torch.float64, device="cuda")
        rt = ops.param(p2, n, False)
        rows = np.arange(C), np.array(at)
        if dist == "gamma":
            _run_gamma(ops, impl, n, x, ops.param(p1, n, False), n, rt, n, out, 0)
            ref, mag = _gamma_terms(x[rows], p1[rows], p2[rows])
        else:
            _run_poisson(ops, impl, n, x, rt, n, out, 0)
            ref, mag = _poisson_terms(x[rows], p2[rows])
        _check(_host(out), ref, mag, f"{dist} {impl} n={n} edges {edges}")


# ----------------------------------------------------------------------------- 2. Normal from ss, const, domain
@pytest.mark.parametrize("impl", IMPLS)
@pytest.mark.parametrize("C", (127, 128, 129, 4097))
def test_logp_normal_ss(impl, C):
    """0.5 (dim log s + log|P| - dim log 2 pi - s ss) per chain; scalar / logdet NULL mean 1 and 0 (128-thread grid)."""
    import torch

    from openmcmc_b200 import kernels as K

    rng = np.random.default_rng(C)
    ss, s, ld = rng.uniform(0.0, 3e3, C), rng.uniform(0.01, 20.0, C), rng.normal(0.0, 40.0, C)
    prefill = rng.normal(0.0, 100.0, C)
    for dim in (1.0, 7.0, 1e6):
        for with_s in (False, True):
            for with_ld in (False, True):
                for acc in (0, 1):
                    ops = _Ops(C)
                    out = _t(prefill) if acc else torch.full((C,), NAN, dtype=torch.float64, device="cuda")
                    args = (C, dim, K.vec(ops.dev(ss), 1), K.vec(ops.dev(s), 1) if with_s else K.vec(None),
                            K.vec(ops.dev(ld), 1) if with_ld else K.vec(None), out, acc)
                    ops.run(impl, lambda: K.logp_normal_ss(*args), K.fop_logp_normal_ss(*args))
                    sc, lg = (s if with_s else np.ones(C)), (ld if with_ld else np.zeros(C))
                    ref = 0.5 * (dim * np.log(sc) + lg - dim * np.log(2 * np.pi) - sc * ss)   # oracle/dist.py:18-20
                    mag = 0.5 * (np.abs(dim * np.log(sc)) + np.abs(lg) + dim * np.log(2 * np.pi) + sc * ss)
                    if acc:
                        ref, mag = ref + prefill, mag + np.abs(prefill)
                    _check(_host(out), ref, mag, f"normal_ss {impl} C={C} dim={dim} s={with_s} ld={with_ld} acc={acc}")


@pytest.mark.parametrize("impl", IMPLS)
def test_logp_const(impl):
    """out = v, or out + v with accumulate: exactly one rounding."""
    import torch

    from openmcmc_b200 import kernels as K

    for C in (1, 127, 128, 129, 4097):
        prefill = np.random.default_rng(C).normal(0.0, 10.0, C)
        for acc in (0, 1):
            ops = _Ops(C)
            out = _t(prefill) if acc else torch.full((C,), NAN, dtype=torch.float64, device="cuda")
            v = -1234.0625 / 3.0
            ops.run(impl, lambda: K.logp_const(v, C, out, acc), K.fop_logp_const(v, C, out, acc))
            assert np.array_equal(_host(out), prefill + v if acc else np.full(C, v)), (impl, C, acc)


@pytest.mark.parametrize("n", (1, 5, 33, 300))
def test_logp_domain(n):
    """A value on a bound is inside (out keeps its sentinel); one element outside, first or last, gives -inf; bounds of
    length 1 or n_elem, per chain; lower bound only, upper bound only."""
    from openmcmc_b200 import kernels as K

    C = 257
    rng = np.random.default_rng(n)
    for lo_len in sorted({1, n}):
        for hi_len in sorted({1, n}):
            for which in ("both", "lower", "upper"):
                lo = rng.uniform(-2.0, -1.0, (C, lo_len))
                hi = rng.uniform(1.0, 2.0, (C, hi_len))
                lo_f, hi_f = np.broadcast_to(lo, (C, n)), np.broadcast_to(hi, (C, n))
                x = rng.uniform(-0.9, 0.9, (C, n))
                case = np.arange(C) % 5        # 0 inside, 1 on the bounds, 2 below at 0, 3 above at n-1, 4 below at n-1
                on = case == 1
                if which != "upper":
                    x[on, 0] = lo_f[on, 0]
                if which == "upper" or (which == "both" and n > 1):
                    x[on, n - 1] = hi_f[on, n - 1]
                x[case == 2, 0] = np.nextafter(lo_f[case == 2, 0], -INF)
                x[case == 3, n - 1] = np.nextafter(hi_f[case == 3, n - 1], INF)
                x[case == 4, n - 1] = lo_f[case == 4, n - 1] - 1.0
                ops = _Ops(C)
                out = ops.dev(np.full(C, 3.25))
                lower = K.vec(ops.dev(lo), lo_len) if which != "upper" else K.vec(None)
                upper = K.vec(ops.dev(hi), hi_len) if which != "lower" else K.vec(None)
                K.logp_domain(C, n, K.vec(ops.dev(x), n), lower, lo_len, upper, hi_len, out)
                below = (x < lo_f).any(axis=1) if which != "upper" else np.zeros(C, bool)
                above = (x > hi_f).any(axis=1) if which != "lower" else np.zeros(C, bool)
                want = np.where(below | above, -INF, 3.25)
                assert np.array_equal(_host(out), want), (n, lo_len, hi_len, which)
                assert (want[case == 1] == 3.25).all() and (want[case == 2] == -INF).all() == (which != "upper")
                assert (want[case == 3] == -INF).all() == (which != "lower")


# ----------------------------------------------------------------------------- 3. sum_log, log_elements, logdet, combine
@pytest.mark.parametrize("n", (1, 255, 256, 257, 100_000))
def test_sum_log(n):
    """sum_i log x_i per matrix; a 0 element gives -inf, a negative one NaN, and the other matrices stay exact."""
    import torch

    from openmcmc_b200 import kernels as K

    rng = np.random.default_rng(n)
    x = np.exp(rng.uniform(-30.0, 30.0, (5, n)))
    x[1, n // 2] = 0.0
    x[3, n - 1] = -0.5
    out = torch.full((5,), NAN, dtype=torch.float64, device="cuda")
    dx = _t(x)
    K.sum_log(dx, n, out)
    with np.errstate(all="ignore"):
        terms = np.log(x)
    ref, mag = _chain_sums(terms, np.abs(terms))
    _check(_host(out), ref, mag, f"sum_log n={n}")
    assert np.isneginf(ref[1]) and np.isnan(ref[3])


@pytest.mark.parametrize("n", (1, 255, 256, 257, 100_000, 1_100_003))
def test_log_elements(n):
    """out = log x element-wise; above 4096 blocks of 256 the grid-stride loop runs more than once."""
    import torch

    from openmcmc_b200 import kernels as K

    rng = np.random.default_rng(n)
    x = np.exp(rng.uniform(-700.0, 700.0, n))
    x[0] = 0.0
    x[-1] = -1.0 if n > 1 else x[-1]
    x[n // 2] = 1.0 if n > 2 else x[n // 2]
    dx = _t(x)
    out = torch.full((n,), NAN, dtype=torch.float64, device="cuda")
    K.log_elements(dx, out)
    with np.errstate(all="ignore"):
        ref = np.log(x)
    _check(_host(out), ref, np.abs(ref), f"log_elements n={n}")


def _spd(n, cond, rng):
    q, _ = np.linalg.qr(rng.standard_normal((n, n)))
    d = np.geomspace(1.0, 1.0 / cond, n) * rng.uniform(0.5, 2.0)
    return (q * d) @ q.T, d


@pytest.mark.parametrize("n", (1, 2, 63, 64))
def test_logdet_dense(n):
    """log|P| by the unblocked Cholesky of one matrix per CTA (n = 64 fills 32 KB of shared memory) against slogdet,
    condition numbers 1 to 1e8; a non-PD matrix in the batch gives NaN and its neighbours stay exact.
    Tolerance: 8 eps (sum_j |log d_j| + n cond), the backward error of a Cholesky seen through log|P|."""
    import torch

    from openmcmc_b200 import kernels as K

    rng = np.random.default_rng(n)
    conds = (1.0, 1e2, 1e4, None, 1e6, 1e8)
    mats, mags = [], []
    for cond in conds:
        if cond is None:                                 # one negative eigenvalue: slogdet's sign is -1
            P, d = _spd(n, 10.0, rng)
            q, _ = np.linalg.qr(rng.standard_normal((n, n)))
            d = d.copy()
            d[0] = -d[0]
            P = (q * d) @ q.T
        else:
            P, d = _spd(n, cond, rng)
        P = 0.5 * (P + P.T)
        mats.append(P)
        mags.append(np.sum(np.abs(np.log(np.abs(d)))) + n * (cond or 1.0))
    Ps = np.stack(mats)
    out = torch.full((len(conds),), 0.0, dtype=torch.float64, device="cuda")
    K.logdet_dense(_t(Ps), n, out)
    sign, ld = np.linalg.slogdet(Ps)
    ref = np.where(sign > 0, ld, NAN)
    assert np.isnan(ref[3])
    _check(_host(out), ref, mags, f"logdet n={n}")


@pytest.mark.parametrize("n_terms", (1, 2, 3, 4))
def test_combine(n_terms):
    """out[c][i] = sum_t s_t[c] x_t[c][i]: scales NULL, shared or per chain; x shared or per chain; out aliasing x0;
    len 0 writes nothing; C len above 16 SMs x 256, so that the grid-stride loop runs more than once."""
    import torch

    from openmcmc_b200 import kernels as K

    big = 16 * torch.cuda.get_device_properties(0).multi_processor_count * 256
    rng = np.random.default_rng(n_terms)
    for C, L in ((1, 1), (7, 33), (3, 257), (7, big // 7 + 1001)):
        xs = [rng.normal(0.0, 10.0, (C, L)) for _ in range(n_terms)]
        ss = [rng.normal(0.0, 3.0, C) for _ in range(n_terms)]
        for scale_mode in ("none", "shared", "per_chain"):
            for x_shared in (False, True):
                for alias in (False, True):
                    ops = _Ops(C)
                    # shared x: the odd terms (term 0 too when it is the only one and out does not alias it)
                    sh = [x_shared and (t % 2 == 1 or (n_terms == 1 and not alias)) for t in range(n_terms)]
                    xf = [np.broadcast_to(x[:1], (C, L)) if sh[t] else x for t, x in enumerate(xs)]
                    sf = [np.ones(C) if scale_mode == "none" else np.full(C, s[0]) if scale_mode == "shared" else s
                          for s in ss]
                    dxs = [ops.dev(x[0] if sh[t] else x) for t, x in enumerate(xs)]
                    vx = [K.vec(d) if sh[t] else K.vec(d, L) for t, d in enumerate(dxs)]
                    vs = [None if scale_mode == "none" else K.vec(ops.dev(s[:1])) if scale_mode == "shared"
                          else K.vec(ops.dev(s), 1) for s in ss]
                    out = dxs[0] if alias else ops.dev(np.full((C, L), NAN))
                    K.combine(C, L, vx, vs, out)
                    ref = sum(s[:, None] * x for s, x in zip(sf, xf))
                    mag = sum(np.abs(s[:, None] * x) for s, x in zip(sf, xf))
                    _check(_host(out), ref, mag, f"combine C={C} L={L} {scale_mode} x_shared={x_shared} alias={alias}")
    out = _t(np.full((3, 4), 7.5))
    K.combine(3, 0, [K.vec(_t(np.zeros((3, 4))), 4)], [None], out)
    assert np.array_equal(_host(out), np.full((3, 4), 7.5))


# ----------------------------------------------------------------------------- 4. linear predictor
def _takes_rows_kernel(terms):
    """The dispatch condition of omc_linear_predictor (logp.cu): one term, even 2 <= p <= 64, 16-byte aligned X, even
    X chain stride."""
    if len(terms) != 1:
        return False
    xv, _, p, _ = terms[0]
    return 2 <= p <= 64 and p % 2 == 0 and xv.ptr % 16 == 0 and xv.chain_stride % 2 == 0


def _predict(kernel, C, n, specs, residual=None, seed=0):
    """specs: (p, transform_exp, layout) per term, layout 'per_chain', 'shared', 'offset' (X one double into its buffer)
    or 'odd_stride' (per-chain X with one padding double); residual: None, 'per_chain' or 'shared'."""
    import torch

    from openmcmc_b200 import kernels as K

    rng = np.random.default_rng(seed)
    ops = _Ops(C)
    terms, ref, mag = [], np.zeros((C, n)), np.zeros((C, n))
    for p, tr, layout in specs:
        X = rng.normal(0.0, 1.0, (C, n, p))
        th = rng.uniform(-1.0, 1.0, (C, p)) if tr else rng.normal(0.0, 2.0, (C, p))
        if layout == "shared":
            X[:] = X[0]
            dX = ops.dev(X[0])
            xv = K.vec(dX)
        elif layout == "offset":
            buf = ops.dev(np.concatenate([[NAN], X.ravel()]))
            xv = K.Vec(buf.data_ptr() + 8, n * p)
        elif layout == "odd_stride":
            pad = np.concatenate([X.reshape(C, n * p), np.full((C, 1), NAN)], axis=1)
            xv = K.vec(ops.dev(pad), n * p + 1)
        else:
            xv = K.vec(ops.dev(X), n * p)
        terms.append((xv, K.vec(ops.dev(th), p), p, tr))
        coef = np.exp(th) if tr else th
        ref += np.einsum("cnp,cp->cn", X, coef)
        mag += np.einsum("cnp,cp->cn", np.abs(X), np.abs(coef))
    assert _takes_rows_kernel(terms) == (kernel == "rows"), "the case does not reach the kernel it names"
    res = None
    if residual is not None:
        r = rng.normal(0.0, 5.0, (C, n))
        if residual == "shared":
            r[:] = r[0]
            res = K.vec(ops.dev(r[0]))
        else:
            res = K.vec(ops.dev(r), n)
        ref, mag = r - ref, mag + np.abs(r)
    out = ops.dev(np.full((C, n), NAN))
    K.linear_predictor(C, n, terms, out, residual_of=res)
    _check(_host(out), ref, mag, f"{kernel} predictor C={C} n={n} {specs} residual={residual}")


@pytest.mark.parametrize("p", (2, 4, 16, 62, 64))
def test_predictor_rows_kernel(p):
    """linear_predictor_rows_kernel: 16 rows per warp, two columns per lane; n around the 16-row block, shared X with
    theta per chain, transform_exp, residual per chain and shared."""
    for n in (1, 15, 16, 17, 1000):
        for layout in ("per_chain", "shared"):
            for tr in (False, True):
                for residual in (None, "per_chain", "shared"):
                    _predict("rows", 3, n, [(p, tr, layout)], residual, seed=p * 1000 + n)


def test_predictor_rows_kernel_grid_stride():
    """C ceil(n/16) warps above the grid cap of 16 CTAs per SM: every warp takes more than one block of rows."""
    _predict("rows", 4, 100_000, [(8, False, "per_chain")], "per_chain", seed=1)


@pytest.mark.parametrize("p", (1, 3, 63, 65, 200))
def test_predictor_generic_kernel(p):
    """linear_predictor_kernel: one warp per output row, odd p and p above 64."""
    for n in (1, 17, 300):
        for layout in ("per_chain", "shared"):
            for tr in (False, True):
                for residual in (None, "per_chain", "shared"):
                    _predict("generic", 3, n, [(p, tr, layout)], residual, seed=p * 1000 + n)


@pytest.mark.parametrize("specs", [
    [(4, False, "per_chain"), (3, True, "shared")],
    [(8, True, "per_chain"), (1, False, "per_chain"), (65, False, "shared")],
    [(2, False, "shared"), (5, True, "per_chain"), (16, True, "per_chain"), (40, False, "per_chain")],
], ids=("generic_2terms", "generic_3terms", "generic_4terms"))
def test_predictor_generic_kernel_terms(specs):
    """2 to 4 terms of different p and mixed transform_exp: the generic kernel."""
    for residual in (None, "per_chain"):
        _predict("generic", 5, 37, specs, residual, seed=len(specs))


@pytest.mark.parametrize("layout", ("offset", "odd_stride"), ids=("generic_unaligned_X", "generic_odd_chain_stride"))
@pytest.mark.parametrize("p", (2, 16, 64))
def test_predictor_generic_kernel_fallback(layout, p):
    """Even p that must leave the rows kernel: X one double into its buffer (not 16-byte aligned), odd X chain stride."""
    for n in (1, 17, 300):
        _predict("generic", 3, n, [(p, False, layout)], "per_chain", seed=p + n)


# ----------------------------------------------------------------------------- 5. the fused store epilogue and copies
def _epilogue(C, wide, it, max_iter, ring, seed):
    """One fused_small launch as the engine builds it: ng_draw (debug_g injected), logp_gamma of its draws, a diagonal
    quadratic form with zero entries, normal_ss on its ss, const, store copies of log_post (count = C) and of the
    quadratic form's [C, p] input (count != C).  Checks every output; returns nothing."""
    import torch

    from openmcmc_b200 import kernels as K
    from oracle import conjugate

    rng = np.random.default_rng(seed)
    ne, pq = 3, (40 if wide else 4)
    ops = _Ops(C)
    a0, b0 = rng.uniform(0.5, 3.0, ne), rng.uniform(0.0, 2.0, 1)
    ss_in, cnt_in = rng.uniform(0.0, 50.0, (C, ne)), rng.integers(0, 30, (C, ne)).astype(np.float64)
    g = rng.gamma(2.0, 1.0, (C, ne))
    sh, rt = rng.uniform(0.5, 4.0, 1), rng.uniform(0.3, 3.0, 1)
    x, mu = rng.normal(0.0, 1.0, (C, pq)), rng.normal(0.0, 1.0, (C, pq))
    Pd = rng.uniform(0.1, 2.0, (C, pq))
    Pd[:, ::3] = 0.0
    s, ld = rng.uniform(0.1, 5.0, C), rng.normal(0.0, 10.0, C)
    konst = -17.125
    draws = ops.dev(np.full((C, ne), NAN))
    lp = ops.dev(np.full(C, NAN))
    qss, qcnt = ops.dev(np.full(C, NAN)), ops.dev(np.full(C, NAN))
    dx = ops.dev(x)
    store_lp, store_x = ops.dev(np.full((max_iter, C), 9.5)), ops.dev(np.full((max_iter, C * pq), 9.5))
    counter = torch.tensor([it], dtype=torch.int64, device="cuda")
    fops = [
        K.fop_ng_draw(C, K.vec(ops.dev(a0)), K.vec(ops.dev(b0)), K.vec(ops.dev(ss_in), ne), K.vec(ops.dev(cnt_in), ne),
                      draws, K.rng(seed=3), debug_g=ops.dev(g), n_elem=ne, a0_len=ne, b0_len=1, ss_stride=1,
                      cnt_stride=1),
        K.fop_logp_gamma(C, ne, K.vec(draws, ne), K.vec(ops.dev(sh)), 1, K.vec(ops.dev(rt)), 1, lp, 0),
        K.fop_quadform(C, pq, K.vec(dx, pq), K.vec(ops.dev(mu), pq), K.MAT_DIAG, K.vec(ops.dev(Pd), pq), qss, qcnt),
        K.fop_logp_normal_ss(C, pq, K.vec(qss, 1), K.vec(ops.dev(s), 1), K.vec(ops.dev(ld), 1), lp, 1),
        K.fop_logp_const(konst, C, lp, 1),
        K.fop_store_copy(lp, store_lp, C, counter, max_iter, ring),
        K.fop_store_copy(dx, store_x, C * pq, counter, max_iter, ring),
    ]
    K.fused_small(C, fops)()
    d = _host(draws)
    for c in range(C):
        for k in range(ne):
            ref, _, _ = conjugate.normal_gamma(a0[k], b0[0], ss_in[c, k], cnt_in[c, k], g[c, k])
            assert abs(d[c, k] - ref) <= 1e-12 * abs(ref), (C, wide, c, k, d[c, k], ref)
    qref = np.array([conjugate.quadform(Pd[c], x[c], mu[c]) for c in range(C)])
    q = _host(qss)
    _check(q, qref[:, 0], np.sum(Pd * (x - mu) ** 2, axis=1), f"quadform C={C} wide={wide}")
    assert np.array_equal(_host(qcnt), qref[:, 1]) and (qref[:, 1] < pq).all()
    glp, gmag = _chain_sums(*_gamma_terms(d, np.full_like(d, sh[0]), np.full_like(d, rt[0])))
    nref = 0.5 * (pq * np.log(s) + ld - pq * np.log(2 * np.pi) - s * q)       # oracle/dist.py:18-20 on the device's ss
    nmag = 0.5 * (np.abs(pq * np.log(s)) + np.abs(ld) + pq * np.log(2 * np.pi) + s * q)
    ref = np.array([math.fsum(v) for v in zip(glp, nref, np.full(C, konst))])
    got = _host(lp)
    _check(got, ref, gmag + nmag + abs(konst), f"log_post C={C} wide={wide}")
    row = it % max_iter if ring else it
    want_lp, want_x = np.full((max_iter, C), 9.5), np.full((max_iter, C * pq), 9.5)
    if ring or it < max_iter:
        want_lp[row], want_x[row] = got, x.ravel()
    assert np.array_equal(_host(store_lp), want_lp), (C, wide, it, max_iter, ring)
    assert np.array_equal(_host(store_x), want_x), (C, wide, it, max_iter, ring)


COUNTER_CASES = [(0, 6, False), (3, 6, False), (5, 6, False), (6, 6, False), (11, 6, False),
                 (0, 4, True), (5, 4, True), (11, 4, True)]


@pytest.mark.parametrize("wide", (False, True), ids=("fused_1lane", "fused_32lanes"))
@pytest.mark.parametrize("C", (1, 5, 129, 1000))
def test_fused_store_epilogue(C, wide):
    for it, max_iter, ring in COUNTER_CASES:
        _epilogue(C, wide, it, max_iter, ring, seed=C + it)


def test_fused_copy_of_a_produced_array_is_refused():
    """A copy of count != C whose source another op of the same launch writes would race with it: refused."""
    from openmcmc_b200 import _cabi
    from openmcmc_b200 import kernels as K

    import torch

    C, ne = 5, 3
    ops = _Ops(C)
    lp, draws = ops.dev(np.zeros(C)), ops.dev(np.zeros((C, ne)))
    counter = torch.zeros(1, dtype=torch.int64, device="cuda")
    dst = ops.dev(np.zeros((4, 2 * C * ne)))
    ng = K.fop_ng_draw(C, K.vec(ops.dev(np.ones(1))), K.vec(ops.dev(np.ones(1))), K.vec(ops.dev(np.ones((C, ne))), ne),
                       K.vec(ops.dev(np.ones((C, ne))), ne), draws, K.rng(seed=1), n_elem=ne, ss_stride=1, cnt_stride=1)
    for producer, src, count in ((K.fop_logp_const(1.0, C, lp, 0), lp, C + 1),
                                 (ng, draws, C * ne)):
        with pytest.raises(_cabi.OmcError, match="produced by op 0"):
            K.fused_small(C, [producer, K.fop_store_copy(src, dst, count, counter, 4)])()
    K.fused_small(C, [K.fop_logp_const(1.0, C, lp, 0), K.fop_store_copy(lp, dst, C, counter, 4)])()   # count = C: fine
    assert np.array_equal(_host(dst)[0, :C], np.ones(C))


@pytest.mark.parametrize("count", (1, 255, 256, 400_003))
def test_store_copy_standalone(count):
    """omc_store_copy / omc_store_copy_ring: row it of the store, nothing at or past max_iter, slot it % ring; 400,003
    values take more than one pass of the capped grid."""
    import torch

    from openmcmc_b200 import kernels as K

    src = np.random.default_rng(count).normal(0.0, 1.0, count)
    dsrc = _t(src)
    for it, max_iter, ring in COUNTER_CASES:
        dst = torch.full((max_iter, count), 9.5, dtype=torch.float64, device="cuda")
        counter = torch.tensor([it], dtype=torch.int64, device="cuda")
        K.store_copy(dsrc, dst, count, counter, max_iter, ring)
        want = np.full((max_iter, count), 9.5)
        if ring or it < max_iter:
            want[it % max_iter if ring else it] = src
        assert np.array_equal(_host(dst), want), (count, it, max_iter, ring)
