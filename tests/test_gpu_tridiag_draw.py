"""omc_tridiag_nn_draw element by element against LAPACK, on the kernels a sweep runs.

The draw picks its kernels from its arguments (tridiag.cu, omc_tridiag_nn_draw):
  solve     tg_solve_kernel<GENERAL, DEBUG>: GENERAL when w, h or mu0 is given; DEBUG when debug_z, logdet, probe_l
            or probe_c is given, or x is NULL.  Only DEBUG = 0 draws its own normals.
  aggregate tg_aggregate_kernel<GENERAL, G>: G = 2 chains per CTA when not GENERAL and C >= 2, else G = 1.
Every case id names the pair it reaches as solve<GENERAL,DEBUG>-agg<GENERAL,G>.

Reference, per chain: Q = lam P + tau W as a band, scipy.linalg.cholesky_banded (the factor, compared with
probe_l / probe_c), cho_solve_banded (the mean), solve_banded on L' (x = mu + L^-T z).  Bars: factor and mean rel
1e-10, x 1e-9, log-determinant rel 1e-11, quadratic forms |got - ref| <= 64 eps M with M the sum of the magnitudes
of the per-element addends (exact enough in long double), recomputed from the kernel's own x.

The production kernels (DEBUG = 0) are checked through z = L'(x - mu), recovered from their x with the reference
factor: it must not depend on the data or on n, launches must be bit-reproducible and shardable, and z must match
oracle/tridiag_stream.py, the numpy restatement of the kernel's stream (2e-5 + 2^-21 / r on fp32-assisted pairs of
radius r, 1e-9 on the fp64 redo pairs; the oracle's docstring derives the bar).
"""

import numpy as np
import pytest
from scipy.linalg import cho_solve_banded, cholesky_banded, solve_banded

from oracle import tridiag_stream as ts

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps
SEED, SITE = 9, 1            # the production draws at 64 x 1e6 take 27 redo pairs with this seed (sweep 0)
N_BIG, C_BIG = 1_000_000, 64


def _kernels(C, general, debug):
    g = 1 if general or C < 2 else 2
    return f"solve<{int(general)},{int(debug)}>-agg<{int(general)},{g}>"


def _grid(n):
    """bench.build_gmrf's grid: regular s_i = i 60/99, RW1 precision, P[0,0] += 1e-3."""
    if n == 1:
        return np.array([1.0 + 1e-3]), np.zeros(0)
    dr = 1.0 / np.diff(np.arange(n) * (60.0 / 99.0))
    pd = np.append(np.append(dr[0], dr[:-1] + dr[1:]), dr[-1])
    pd[0] += 1e-3
    return pd, -dr


def _truth(n):
    s = np.arange(n) * (60.0 / 99.0)
    return np.sin(s / 20) + 2 * np.cos(s / 12) + 2


def _matvec(pd, pe, v):
    out = pd * v
    out[:-1] += pe * v[1:]
    out[1:] += pe * v[:-1]
    return out


def _dev(a):
    import torch

    return torch.as_tensor(np.array(a, dtype=np.float64)).cuda()


def _reference(pd, pe, lam, tau, w, y, h):
    """Band Cholesky factor (row 0 diagonal, row 1 sub-diagonal) and mean of Q = lam P + tau W, b = lam h + tau W y."""
    n = pd.size
    ab = np.zeros((2, n))
    ab[0] = lam * pd + tau * w
    ab[1, : n - 1] = lam * pe
    cb = cholesky_banded(ab, lower=True, check_finite=False)
    b = tau * w * y + (lam * h if h is not None else 0.0)
    return cb, cho_solve_banded((cb, True), b, check_finite=False)


def _lt_solve(cb, z):
    """L^-T z."""
    u = np.zeros_like(cb)
    u[0, 1:] = cb[1, :-1]
    u[1] = cb[0]
    return solve_banded((0, 1), u, z, check_finite=False)


def _lt_mul(cb, v):
    """L' v."""
    z = cb[0] * v
    z[:-1] += cb[1, :-1] * v[1:]
    return z


def _ss_err(got, x, pd, pe, mu0, y, w):
    """(|got - ref| / (64 eps M)) for ss_prior and ss_lik of the kernel's own x, in long double."""
    ld = np.longdouble
    r = x - mu0 if mu0 is not None else x                  # rounded in fp64 as the kernel rounds it
    q = y - x
    tp = pd.astype(ld) * r * r
    to = 2 * pe.astype(ld) * r[:-1] * r[1:]
    tl = (w.astype(ld) if w is not None else ld(1)) * q * q
    out = []
    for g, terms in zip(got, ((tp, to), (tl,))):
        ref = sum(t.sum() for t in terms)
        m = sum(np.abs(t).sum() for t in terms)
        out.append(float(abs(ld(g) - ref) / (64 * EPS * m)) if m > 0 else abs(g))
    return out


class Problem:
    """One omc_tridiag_nn_draw problem on the device: grid, data, per-chain lam / tau and optional w / mu0 / h."""

    def __init__(self, C, n, seed, weighted=False, with_mu=False, y_mode="rows"):
        import torch

        from openmcmc_b200 import kernels as K

        K.init_device()
        rng = np.random.default_rng(seed)
        self.C, self.n = C, n
        self.pd, self.pe = _grid(n)
        self.lam = 10.0 ** rng.uniform(1, 3, C)
        self.tau = rng.uniform(0.3, 3, C)
        self.w = rng.uniform(0.5, 1.5, (C, n)) if weighted else None
        self.mu0 = rng.standard_normal(n) + 1 if with_mu else None
        self.h = _matvec(self.pd, self.pe, self.mu0) if with_mu else None
        truth = _truth(n)
        if y_mode == "shared":
            self.y = np.broadcast_to(truth + rng.standard_normal(n), (C, n))
        else:
            self.y = truth + rng.standard_normal((C, n))
        self.d_pd, self.d_pe = _dev(self.pd), _dev(self.pe)
        self.d_lam, self.d_tau = _dev(self.lam), _dev(self.tau)
        if y_mode == "shared":
            self.d_y = _dev(self.y[0])
            yv = K.vec(self.d_y)
        elif y_mode == "unaligned":   # every chain at an odd double offset: chain_stride n + 1 (n odd), element 1 first
            assert n % 2 == 1
            buf = torch.zeros(1 + C * (n + 1), dtype=torch.float64, device="cuda")
            buf[1:].view(C, n + 1)[:, :n] = _dev(self.y)
            self.d_y = buf[1:]
            yv = K.vec((self.d_y, n + 1))
        else:
            self.d_y = _dev(self.y)
            yv = K.vec(self.d_y, n)
        self.d_w = _dev(self.w) if weighted else None
        self.d_mu, self.d_h = (_dev(self.mu0), _dev(self.h)) if with_mu else (None, None)
        self.common = dict(lam=K.vec(self.d_lam, 1), tau=K.vec(self.d_tau, 1), y=yv,
                           w=K.vec(self.d_w, n) if weighted else None, mu0=K.vec(self.d_mu) if with_mu else None,
                           h=K.vec(self.d_h) if with_mu else None)
        self.general = weighted or with_mu
        self.ws = torch.zeros(K.tridiag_workspace(C, n), dtype=torch.uint8, device="cuda")

    def draw(self, **kw):
        from openmcmc_b200 import kernels as K

        K.tridiag_nn_draw(K.tridiag_args(self.C, self.n, self.d_pd, self.d_pe, self.ws, **self.common, **kw))

    def out(self, *shape):
        import torch

        return torch.zeros(*shape, dtype=torch.float64, device="cuda")

    def chain(self, c):
        """Reference factor and mean of chain c, and its (w, mu0, h) operands."""
        w = self.w[c] if self.w is not None else np.ones(self.n)
        cb, mu = _reference(self.pd, self.pe, self.lam[c], self.tau[c], w, self.y[c], self.h)
        return cb, mu

    def ss_err(self, c, x, ss_prior, ss_lik):
        return _ss_err((ss_prior, ss_lik), x, self.pd, self.pe, self.mu0, self.y[c],
                       self.w[c] if self.w is not None else None)


def _injected(P, z, sweeps=1):
    """Injected-z draws (DEBUG solve kernel) with every probe, `sweeps` consecutive draws on one workspace with the
    sweep counter advanced between them as a graph replay advances it; then checks every chain of every draw."""
    import torch

    from openmcmc_b200 import kernels as K

    C, n = P.C, P.n
    d_z = _dev(z)                           # [sweeps, C, n]
    sweep = torch.zeros(1, dtype=torch.int64, device="cuda")
    status = torch.zeros(C, dtype=torch.int32, device="cuda")
    res = []
    for s in range(sweeps):
        r = dict(x=P.out(C, n), ss_prior=P.out(C), ss_lik=P.out(C), logdet=P.out(C), probe_l=P.out(C, n),
                 probe_c=P.out(C, max(n - 1, 1)))
        P.draw(**r, debug_z=d_z, debug_sweep_stride=C * n, rng_=K.rng(seed=1, sweep=sweep, site=SITE), status=status)
        K.counter_add(sweep)
        res.append(r)
    mean = P.out(C, n)
    P.draw(x=mean, debug_z=torch.zeros(C, n, dtype=torch.float64, device="cuda"))
    torch.cuda.synchronize()
    assert status.cpu().tolist() == [0] * C
    mean = mean.cpu().numpy()
    res = [{k: v.cpu().numpy() for k, v in r.items()} for r in res]
    for c in range(C):
        cb, mu = P.chain(c)
        np.testing.assert_allclose(mean[c], mu, rtol=1e-10, atol=1e-12)
        for s, r in enumerate(res):
            np.testing.assert_allclose(r["probe_l"][c], cb[0], rtol=1e-10)
            np.testing.assert_allclose(r["probe_c"][c, : n - 1], cb[1, : n - 1], rtol=1e-10)
            np.testing.assert_allclose(r["logdet"][c], 2 * np.sum(np.log(cb[0])), rtol=1e-11)
            np.testing.assert_allclose(r["x"][c], mu + _lt_solve(cb, z[s, c]), rtol=1e-9, atol=1e-11)
            assert max(P.ss_err(c, r["x"][c], r["ss_prior"][c], r["ss_lik"][c])) <= 1.0, (s, c)


# ------------------------------------------------------------------------------- a. injected z on every edge
EDGE_N = [1, 2, 17, 18, 19, 35, 36, 37, 2303, 2304, 2305, 4608, 6911, 6912, 6913]


@pytest.mark.parametrize("n,C", [(n, C) for n in EDGE_N for C in (1, 3)],
                         ids=[f"{_kernels(C, False, True)}-n{n}-C{C}" for n in EDGE_N for C in (1, 3)])
def test_injected_tile_and_thread_edges(n, C):
    P = Problem(C, n, seed=n * 10 + C)
    _injected(P, np.random.default_rng(n).standard_normal((1, C, n)))


FORMS = [(False, False), (True, False), (False, True), (True, True)]   # (w, mu0 with h = P mu0)


@pytest.mark.parametrize("n", [2304, 2305, 6913])
@pytest.mark.parametrize("weighted,with_mu", FORMS,
                         ids=[f"{_kernels(3, w or m, True)}-{'w' if w else ''}{'mu0' if m else ''}{'' if w or m else 'plain'}"
                              for w, m in FORMS])
def test_injected_general_forms(weighted, with_mu, n):
    P = Problem(3, n, seed=n + 7, weighted=weighted, with_mu=with_mu)
    assert P.general == (weighted or with_mu)
    _injected(P, np.random.default_rng(n + 1).standard_normal((1, 3, n)))


@pytest.mark.parametrize("y_mode,n", [("unaligned", 6913), ("shared", 6912)],
                         ids=[f"{_kernels(3, False, True)}-y_stride_n+1", f"{_kernels(3, False, True)}-y_shared"])
def test_injected_y_layouts(y_mode, n):
    P = Problem(3, n, seed=11, y_mode=y_mode)
    _injected(P, np.random.default_rng(12).standard_normal((1, 3, n)))


@pytest.mark.parametrize("weighted", [False, True],
                         ids=[_kernels(3, False, True), _kernels(3, True, True)])
def test_injected_three_sweeps_one_workspace(weighted):
    P = Problem(3, 4609, seed=13, weighted=weighted)
    _injected(P, np.random.default_rng(14).standard_normal((3, 3, 4609)), sweeps=3)


# ------------------------------------------------------------------------------- b/c. the bench shape, 64 x 1e6
@pytest.fixture(scope="module")
def big():
    """64 x 1e6 (C3): one injected-z draw with every probe, the mean, two production draws and a 32-chain shard with
    chain_offset = 32, all on device; then the per-chain reference and the recovered z of the production draw."""
    import torch

    from openmcmc_b200 import kernels as K

    P = Problem(C_BIG, N_BIG, seed=2026)
    C, n = C_BIG, N_BIG
    z_inj = np.random.default_rng(2027).standard_normal((C, n))
    d_z = _dev(z_inj)
    status = torch.zeros(C, dtype=torch.int32, device="cuda")
    inj = dict(x=P.out(C, n), ss_prior=P.out(C), ss_lik=P.out(C), logdet=P.out(C), probe_l=P.out(C, n),
               probe_c=P.out(C, n - 1))
    P.draw(**inj, debug_z=d_z, status=status)
    mean = P.out(C, n)
    P.draw(x=mean, debug_z=torch.zeros_like(d_z))
    del d_z
    sweep = torch.zeros(1, dtype=torch.int64, device="cuda")
    prod = [dict(x=P.out(C, n), ss_prior=P.out(C), ss_lik=P.out(C)) for _ in range(2)]
    for r in prod:
        P.draw(**r, rng_=K.rng(seed=SEED, sweep=sweep, site=SITE))
    half = C // 2
    ws_half = torch.zeros(K.tridiag_workspace(half, n), dtype=torch.uint8, device="cuda")
    x_half = P.out(half, n)
    K.tridiag_nn_draw(K.tridiag_args(half, n, P.d_pd, P.d_pe, ws_half, lam=K.vec(P.d_lam[half:], 1),
                                     tau=K.vec(P.d_tau[half:], 1), y=K.vec(P.d_y[half:], n), x=x_half,
                                     rng_=K.rng(seed=SEED, sweep=sweep, chain_offset=half, site=SITE)))
    torch.cuda.synchronize()
    out = {"P": P, "status": status.cpu().tolist(),
           "same_x": bool(torch.equal(prod[0]["x"], prod[1]["x"])),
           "same_ss": bool(torch.equal(prod[0]["ss_prior"], prod[1]["ss_prior"])
                           and torch.equal(prod[0]["ss_lik"], prod[1]["ss_lik"])),
           "shard_x": bool(torch.equal(x_half, prod[0]["x"][half:]))}
    del x_half, prod[1]
    inj = {k: v.cpu().numpy() if v.dim() == 1 else v for k, v in inj.items()}
    ssp, ssl = prod[0]["ss_prior"].cpu().numpy(), prod[0]["ss_lik"].cpu().numpy()
    err = {k: np.zeros(C) for k in ("l", "c", "mu", "x", "logdet", "ss_inj", "ss_prod", "z_fast", "z_redo")}
    n_redo = 0
    z_rec = np.empty((C, n))
    for c in range(C):
        cb, mu = P.chain(c)
        rel = lambda got, ref: np.max(np.abs(got - ref) / np.abs(ref))   # noqa: E731
        err["l"][c] = rel(inj["probe_l"][c].cpu().numpy(), cb[0])
        err["c"][c] = rel(inj["probe_c"][c].cpu().numpy(), cb[1, :-1])
        err["mu"][c] = np.max(np.abs(mean[c].cpu().numpy() - mu) / np.maximum(np.abs(mu), 1e-2))
        x = inj["x"][c].cpu().numpy()
        err["x"][c] = np.max(np.abs(x - (mu + _lt_solve(cb, z_inj[c]))) / np.maximum(np.abs(x), 1e-2))
        err["logdet"][c] = abs(inj["logdet"][c] / (2 * np.sum(np.log(cb[0]))) - 1)
        err["ss_inj"][c] = max(P.ss_err(c, x, inj["ss_prior"][c], inj["ss_lik"][c]))
        xp = prod[0]["x"][c].cpu().numpy()
        err["ss_prod"][c] = max(P.ss_err(c, xp, ssp[c], ssl[c]))
        z_rec[c] = _lt_mul(cb, xp - mu)
        zm, redo, tol = ts.chain_normals(SEED, 0, c, SITE, n)
        d = np.abs(z_rec[c] - zm) / tol                  # <= 1 within the bar
        err["z_fast"][c] = d[~redo].max()
        err["z_redo"][c] = d[redo].max() if redo.any() else 0.0
        n_redo += int(redo.sum()) // 2
    out.update(err=err, n_redo=n_redo, z_rec=z_rec)
    return out


def test_bench_shape_injected_solve01_agg02(big):
    """solve<0,1>-agg<0,2> at 64 x 1e6: factor, mean, x, log-determinant and both quadratic forms, every chain."""
    assert _kernels(C_BIG, False, True) == "solve<0,1>-agg<0,2>"
    e = big["err"]
    assert big["status"] == [0] * C_BIG
    assert e["l"].max() <= 1e-10 and e["c"].max() <= 1e-10
    assert e["mu"].max() <= 1e-10
    assert e["x"].max() <= 1e-9
    assert e["logdet"].max() <= 1e-11
    assert e["ss_inj"].max() <= 1.0


def test_bench_shape_production_solve00_agg02_quadforms(big):
    """solve<0,0>-agg<0,2>: the fused ss_prior / ss_lik of the production draw against its own x."""
    assert _kernels(C_BIG, False, False) == "solve<0,0>-agg<0,2>"
    assert big["err"]["ss_prod"].max() <= 1.0


def test_bench_shape_production_solve00_agg02_deterministic_and_shardable(big):
    """Two identical launches are bit-identical; chains 32-63 launched alone with chain_offset = 32 are bit-identical
    to those rows of the 64-chain launch (a different tile-major interleaving of the look-back)."""
    assert big["same_x"] and big["same_ss"]
    assert big["shard_x"]


def test_bench_shape_production_solve00_agg02_z_matches_stream(big):
    """z = L'(x - mu) of the production draw against the restated stream, element by element, on all 64 chains."""
    e = big["err"]
    assert big["n_redo"] >= 10
    assert e["z_fast"].max() <= 1.0, e["z_fast"]
    assert e["z_redo"].max() <= 1.0, e["z_redo"]


def _production(P, x, chain_offset=0, **kw):
    from openmcmc_b200 import kernels as K

    P.draw(x=x, rng_=K.rng(seed=SEED, site=SITE, chain_offset=chain_offset), **kw)


def test_production_solve10_agg11_z_independent_of_data(big):
    """Problem B (other y, lam, tau, weights w and prior mean mu0: the GENERAL kernels) on chains 48-63 of the same
    seed, sweep and site: its recovered z equals problem A's to 1e-9, and its quadratic forms match its own x."""
    C, off, n = 16, 48, N_BIG
    assert _kernels(C, True, False) == "solve<1,0>-agg<1,1>"
    B = Problem(C, n, seed=77, weighted=True, with_mu=True)
    x, ssp, ssl = B.out(C, n), B.out(C), B.out(C)
    _production(B, x, chain_offset=off, ss_prior=ssp, ss_lik=ssl)
    ssp, ssl = ssp.cpu().numpy(), ssl.cpu().numpy()
    for c in range(C):
        cb, mu = B.chain(c)
        xc = x[c].cpu().numpy()
        z = _lt_mul(cb, xc - mu)
        assert np.max(np.abs(z - big["z_rec"][off + c])) <= 1e-9, c
        assert max(B.ss_err(c, xc, ssp[c], ssl[c])) <= 1.0, c


def test_production_solve00_agg02_z_independent_of_n(big):
    """The z recovered from a draw at n = 5000 are the first 5000 z of the 1e6 draw."""
    A = big["P"]
    n = 5000
    S = Problem(C_BIG, n, seed=1)
    S.lam, S.tau, S.y = A.lam, A.tau, A.y[:, :n]
    S.d_lam, S.d_tau, S.d_y = A.d_lam, A.d_tau, _dev(S.y)
    from openmcmc_b200 import kernels as K

    S.common.update(lam=K.vec(S.d_lam, 1), tau=K.vec(S.d_tau, 1), y=K.vec(S.d_y, n))
    x = S.out(C_BIG, n)
    _production(S, x)
    x = x.cpu().numpy()
    for c in range(C_BIG):
        cb, mu = S.chain(c)
        assert np.max(np.abs(_lt_mul(cb, x[c] - mu) - big["z_rec"][c, :n])) <= 1e-9, c


# ------------------------------------------------------------------------------- c. production kernels, small
RAGGED_N, RAGGED_SEED = 5516, 1037118    # found with the model: the pair of elements 5514-5515 is redone (chain 0)


@pytest.mark.parametrize("weighted", [False, True], ids=[_kernels(1, False, False), _kernels(1, True, False)])
def test_production_redo_pair_at_ragged_tile_end(weighted):
    """n = 5516: the last tile holds 908 elements and thread 50 of it 8; its last pair (elements 5514, 5515, block 1531
    words z, w) has a radius word below 2^12, so the device redoes it in fp64.  Every element against the model."""
    import torch

    n = RAGGED_N
    blk, half, _ = ts.element_pair(n - 1)
    assert n % ts.TILE == 908 and (n % ts.TILE) % 18 == 8 and blk == 1531 and half == 1
    z_model, redo, tol = ts.chain_normals(RAGGED_SEED, 0, 0, SITE, n)
    assert redo[n - 2] and redo[n - 1] and redo.sum() == 2
    P = Problem(1, n, seed=5, weighted=weighted)
    x = P.out(1, n)
    from openmcmc_b200 import kernels as K

    P.draw(x=x, rng_=K.rng(seed=RAGGED_SEED, site=SITE))
    torch.cuda.synchronize()
    cb, mu = P.chain(0)
    z = _lt_mul(cb, x[0].cpu().numpy() - mu)
    assert np.max(np.abs(z[-2:] - z_model[-2:])) <= 1e-9
    assert np.all(np.abs(z - z_model) <= tol)


@pytest.mark.parametrize("weighted", [False, True], ids=[_kernels(2, False, False), _kernels(2, True, False)])
def test_production_counter_spill_n_4e6(weighted):
    """C = 2, n = 4e6: Philox block 2^20 (block 1 of group 209,715, first element 3,774,874) is the first whose
    index spills into counter word 1.  Elements 3,774,800-3,775,000 and a random sample beyond, against the model."""
    import torch

    n, C = 4_000_000, 2
    first = 209_715 * 18 + 4
    assert ts.element_pair(first)[0] == 1 << 20 and ts.element_pair(first - 1)[0] == (1 << 20) - 1
    P = Problem(C, n, seed=6, weighted=weighted)
    x = P.out(C, n)
    from openmcmc_b200 import kernels as K

    P.draw(x=x, rng_=K.rng(seed=SEED, site=SITE))
    torch.cuda.synchronize()
    idx = np.concatenate([np.arange(3_774_800, 3_775_001),
                          np.random.default_rng(8).integers(3_775_001, n, 20_000), [n - 1]])
    for c in range(C):
        cb, mu = P.chain(c)
        z = _lt_mul(cb, x[c].cpu().numpy() - mu)[idx]
        zm, redo, tol = ts.normals_at(SEED, 0, c, SITE, idx)
        assert np.all(np.abs(z - zm) <= tol), c


@pytest.mark.parametrize("weighted", [False, True], ids=[_kernels(2, False, False), _kernels(2, True, False)])
def test_production_not_positive_definite_sets_status(weighted):
    """An indefinite P rescued by the likelihood in chain 1 only: the status word flags chain 0 alone (no fault)."""
    import torch

    from openmcmc_b200 import kernels as K

    n, C = 5000, 2
    pd = np.full(n, 2.0)
    pd[3000] = -5.0
    pe = np.full(n - 1, -1.0)
    d_pd, d_pe, d_y, tau = _dev(pd), _dev(pe), _dev(np.ones(n)), _dev(np.array([0.1, 100.0]))
    d_w = _dev(np.ones((C, n))) if weighted else None
    ws = torch.zeros(K.tridiag_workspace(C, n), dtype=torch.uint8, device="cuda")
    x = torch.empty(C, n, dtype=torch.float64, device="cuda")
    status = torch.zeros(C, dtype=torch.int32, device="cuda")
    K.tridiag_nn_draw(K.tridiag_args(C, n, d_pd, d_pe, ws, x=x, tau=K.vec(tau, 1), y=K.vec(d_y),
                                     w=K.vec(d_w, n) if weighted else None, rng_=K.rng(seed=3, site=SITE),
                                     status=status))
    torch.cuda.synchronize()
    assert status.cpu().tolist() == [1, 0]
    assert torch.isfinite(x[1]).all()
