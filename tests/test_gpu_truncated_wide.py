"""GPU parity of the truncated-prior NormalNormal draw for 64 < p <= 512: one coordinate-wise truncated Gibbs scan per
chain, one warp per chain streaming the rows of G (and of a dense P0) through shared memory (trunc_scan.cu).

Everything is checked against the numpy oracle (oracle.gmrf.gibbs_canonical_truncated_normal,
oracle.conjugate.normal_normal_dense_truncated), which the truncreg_* goldens pin against the reference: the gmrf
module function, the kernel through K.nn_dense_draw with per-chain tau / lambda / mu0 and the three prior kinds, whole
MCMC chain replays with injected uniforms and gamma variates, a free-running run against a free-running oracle chain,
sharding invariance of the kernel, a non-PD chain inside a batch, and the refusals above p = 512.  Tolerances as
DESIGN §4: 1e-9 on draws, 1e-10 on deterministic quantities.
"""

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

EYE, DIAG, DENSE = 0, 1, 2


def _bounds(kind, p):
    if kind == "box":
        return np.array([-0.4]), np.array([0.6])
    if kind == "upper":
        return None, np.array([0.3])
    rng = np.random.default_rng(p)
    lo, hi = -0.5 - rng.random(p), 0.5 + rng.random(p)
    lo[::3] = -np.inf
    hi[1::4] = np.inf
    return lo, hi


@pytest.mark.parametrize("bounds", ["box", "vector", "upper"])
@pytest.mark.parametrize("p", [65, 96, 127, 128, 129, 200, 333, 512])
def test_gmrf_gibbs_scan_matches_oracle(p, bounds):
    """gmrf.gibbs_canonical_truncated_normal with injected uniforms == the oracle scan; odd p puts the rows of Q at odd
    doubles (the envelope path of the row copies)."""
    from oracle import gmrf as ogmrf

    from openmcmc_b200 import gmrf

    rng = np.random.default_rng(1000 + p)
    A = rng.standard_normal((p, 2 * p))
    Q = A @ A.T / (2 * p) + 0.5 * np.eye(p)
    b = rng.standard_normal((p, 1))
    x0 = 0.3 * rng.standard_normal((p, 1))
    u = rng.random(p)
    lo, hi = _bounds(bounds, p)
    x = gmrf.gibbs_canonical_truncated_normal(b, Q, x0.copy(), lo, hi, u=u)
    ref = ogmrf.gibbs_canonical_truncated_normal(b, Q, x0, lo, hi, u)
    assert x.shape == (p, 1)
    np.testing.assert_allclose(x, ref, rtol=1e-9, atol=1e-12)
    lo_b = -np.inf if lo is None else np.broadcast_to(lo.reshape(-1), (p,))
    hi_b = np.broadcast_to(hi.reshape(-1), (p,))
    assert np.all(x.ravel() >= lo_b) and np.all(x.ravel() <= hi_b)


def _problem(C, p, kind, shared_P0, seed):
    rng = np.random.default_rng(seed)
    A = rng.standard_normal((C, 2 * p, p))
    G = A.transpose(0, 2, 1) @ A / (2 * p)
    gv = rng.standard_normal((C, p))
    tau = rng.random(C) * 2.0 + 0.5
    lam = rng.random(C) + 0.1
    mu0 = 0.2 * rng.standard_normal((C, p))
    nP = 1 if shared_P0 else C
    if kind == EYE:
        P0 = None if shared_P0 else rng.random((C, 1)) + 0.5
    elif kind == DIAG:
        P0 = rng.random((nP, p)) + 0.5
    else:
        B = rng.standard_normal((nP, p, p))
        P0 = B @ B.transpose(0, 2, 1) / p + np.eye(p)
    x0 = 0.3 * rng.standard_normal((C, p))
    u = rng.random((C, p))
    lo, hi = _bounds("vector", p)
    return dict(C=C, p=p, kind=kind, shared=shared_P0, G=G, gv=gv, tau=tau, lam=lam, mu0=mu0, P0=P0, x0=x0, u=u, lo=lo,
                hi=hi)


def _launch(pr, lam=None, u=True, rng=None, probes=False, chains=None):
    """One omc_nn_dense_draw in truncated mode on pr (or on the chain slice `chains` of it).  Returns beta, status and
    (with probes) Q, b."""
    import torch

    from openmcmc_b200 import kernels as K

    K.init_device(0)
    p = pr["p"]
    sl = slice(0, pr["C"]) if chains is None else chains
    C = sl.stop - sl.start
    d = lambda a: torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device="cuda")  # noqa: E731
    stats = d(np.concatenate([pr["G"][sl].reshape(C, -1), pr["gv"][sl], np.zeros((C, 2))], axis=1))
    P0 = pr["P0"]
    if P0 is None:
        pvec = K.vec(None)
    elif pr["shared"]:
        P0t = d(P0[0].reshape(-1))
        pvec = K.vec(P0t)
    else:
        P0t = d(P0[sl].reshape(C, -1))
        pvec = K.vec(P0t, P0t.shape[1])
    tau, lamt, mu0 = d(pr["tau"][sl]), d((pr["lam"] if lam is None else lam)[sl]), d(pr["mu0"][sl])
    beta = d(pr["x0"][sl])
    lo, hi = d(pr["lo"]), d(pr["hi"])
    du = d(pr["u"][sl]) if u else None
    status = torch.zeros(C, dtype=torch.int32, device="cuda")
    pQ = torch.zeros(C, p * p, dtype=torch.float64, device="cuda") if probes else None
    pb = torch.zeros(C, p, dtype=torch.float64, device="cuda") if probes else None
    K.nn_dense_draw(C, p, stats, K.vec(tau, 1), pr["kind"], pvec, K.vec(lamt, 1), K.vec(mu0, p), beta,
                    rng if rng is not None else K.rng(seed=5, site=3), probe_Q=pQ, probe_b=pb, status=status,
                    trunc=(K.vec(lo), p, K.vec(hi), p), debug_u=du)
    torch.cuda.synchronize()
    out = [beta.cpu().numpy(), status.cpu().numpy()]
    out += [pQ.cpu().numpy().reshape(C, p, p), pb.cpu().numpy()] if probes else [None, None]
    return out


def _oracle(pr, c):
    from oracle import conjugate

    P0 = pr["P0"]
    if P0 is None:
        P0c = np.asarray(1.0)
    else:
        P0c = P0[0 if pr["shared"] else c]
        if pr["kind"] == EYE:
            P0c = np.asarray(float(P0c[0]))
    return conjugate.normal_normal_dense_truncated(pr["G"][c], pr["gv"][c], pr["tau"][c], P0c, pr["lam"][c],
                                                   pr["mu0"][c], pr["x0"][c], pr["lo"], pr["hi"], pr["u"][c])


@pytest.mark.parametrize("shared_P0", [False, True])
@pytest.mark.parametrize("kind", [EYE, DIAG, DENSE])
@pytest.mark.parametrize("p,C", [(129, 37), (150, 300), (512, 200)])
def test_kernel_matches_oracle_per_chain(p, C, kind, shared_P0):
    """K.nn_dense_draw(trunc=...) on many chains, per-chain tau / lambda / mu0, shared or per-chain P0: every sampled
    chain's scan equals the oracle's, probe_Q / probe_b equal the oracle's Q / b.  p = 129 with a per-chain P0 puts
    rows of P0 at odd doubles at the start of a chain and at the end of the array (the plain-load elements)."""
    pr = _problem(C, p, kind, shared_P0, seed=10 * p + kind)
    beta, status, Q, b = _launch(pr, probes=True)
    assert not status.any()
    picks = sorted({0, 1, C // 2, C - 2, C - 1} | set(np.random.default_rng(p).integers(0, C, 3).tolist()))
    for c in picks:
        ref = _oracle(pr, c)
        np.testing.assert_allclose(Q[c], ref["Q"], rtol=1e-10, atol=1e-13)
        np.testing.assert_allclose(b[c], ref["b"].ravel(), rtol=1e-10, atol=1e-13)
        np.testing.assert_allclose(beta[c], ref["x"].ravel(), rtol=1e-9, atol=1e-12)
    assert np.all(beta >= pr["lo"]) and np.all(beta <= pr["hi"])


def _gdict(n, p, seed, prior="eye", lower=None, upper=None, weighted=False):
    """A regression problem in the format of tests/test_gpu_mcmc_regression.build (truncreg golden layout)."""
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, p))
    X[:, 0] = 1.0
    y = X @ (0.3 * rng.standard_normal((p, 1))) + rng.standard_normal((n, 1))
    if prior == "dense":
        B = rng.standard_normal((p, p))
        P = B @ B.T / p + np.eye(p)
    else:
        P = np.eye(p)
    return {"X": X, "y": y, "mu": 0.1 * rng.standard_normal((p, 1)), "w": rng.random(n) + 0.5 if weighted else np.zeros(0),
            "P_lambda": P, "prior": np.array(prior), "order": np.array(["beta", "tau", "lambda"]),
            "lower": np.array([-np.inf]) if lower is None else np.array([lower]),
            "upper": np.array([np.inf]) if upper is None else np.array([upper])}


@pytest.mark.parametrize("p,prior,lower,upper,weighted", [(80, "eye", -0.4, 0.6, False), (200, "dense", None, 0.5, True)])
def test_mcmc_replays_oracle_chain(p, prior, lower, upper, weighted):
    """Whole MCMC run of the truncated regression model with the uniforms of the scan and the gamma variates of tau /
    lambda injected: beta, tau, lambda and log_post equal the oracle chain's."""
    from test_gpu_mcmc_regression import build

    from openmcmc_b200.mcmc import MCMC
    from oracle import conjugate, dist

    n, n_iter = 400, 4
    g = _gdict(n, p, seed=p, prior=prior, lower=lower, upper=upper, weighted=weighted)
    rng = np.random.default_rng(p + 1)
    U = rng.random((n_iter, p))
    gt = rng.standard_gamma(1e-3 + n / 2, size=n_iter)
    gl = rng.standard_gamma(1e-3 + p / 2, size=n_iter)
    mdl, samplers, state = build(g)
    M = MCMC(state, samplers, model=mdl, n_burn=0, n_iter=n_iter,
             debug_draws={"beta": {"u": U}, "tau": {"g": gt}, "lambda": {"g": gl}})
    M.run_mcmc()
    X, y, mu, P0 = g["X"], g["y"], g["mu"], g["P_lambda"]
    w = g["w"] if g["w"].size else None
    logdet_P0 = 2 * np.sum(np.log(np.diag(np.linalg.cholesky(P0))))
    logdet_W = 0.0 if w is None else float(np.sum(np.log(w)))
    lo = None if lower is None else g["lower"]
    hi = None if upper is None else g["upper"]
    s = {"beta": np.zeros((p, 1)), "tau": 1.0, "lambda": 0.01}
    G, gv, _, _ = conjugate.regression_suffstats(X, y, w)
    for it in range(n_iter):
        s["beta"] = conjugate.normal_normal_dense_truncated(G, gv, s["tau"], P0, s["lambda"], mu, s["beta"], lo, hi,
                                                            U[it])["x"]
        _, _, rss, cnt = conjugate.regression_suffstats(X, y, w, s["beta"])
        s["tau"], _, _ = conjugate.normal_gamma(1e-3, 1e-3, rss, cnt, gt[it])
        ss, cnt = conjugate.quadform(P0, s["beta"], mu)
        s["lambda"], _, _ = conjugate.normal_gamma(1e-3, 1e-3, ss, cnt, gl[it])
        _, _, rss, _ = conjugate.regression_suffstats(X, y, w, s["beta"])
        ssb, _ = conjugate.quadform(P0, s["beta"], mu)
        lp = (dist.normal_log_p_from_ss(n, s["tau"], logdet_W, rss) + dist.normal_log_p_from_ss(p, s["lambda"], logdet_P0, ssb)
              + dist.gamma_log_p(s["tau"], 1e-3, 1e-3) + dist.gamma_log_p(s["lambda"], 1e-3, 1e-3))
        np.testing.assert_allclose(M.store["beta"][:, it], s["beta"].ravel(), rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(M.store["tau"][0, it], s["tau"], rtol=1e-9)
        np.testing.assert_allclose(M.store["lambda"][0, it], s["lambda"], rtol=1e-9)
        np.testing.assert_allclose(M.store["log_post"][it, 0], lp, rtol=1e-10)


def test_free_running_stays_inside_and_matches_oracle_chain():
    """Free-running truncated Gibbs at p = 100 (Philox uniforms), 32 chains: every stored draw inside the bounds;
    per-coordinate means agree with a free-running oracle chain (numpy RNG) within Monte-Carlo error."""
    from test_gpu_mcmc_regression import build

    from openmcmc_b200.mcmc import MCMC
    from oracle import conjugate

    p = 100
    g = _gdict(400, p, seed=21, lower=-0.4, upper=0.6)
    mdl, samplers, state = build(g, response=False)
    M = MCMC(state, samplers, model=mdl, n_burn=100, n_iter=200, n_chains=32, seed=11)
    M.run_mcmc()
    b = M.store["beta"]                                      # (C, p, n_iter)
    assert np.all(b >= -0.4) and np.all(b <= 0.6)
    assert np.std(b[:, 0, -1]) > 0
    rng = np.random.default_rng(3)
    X, y, mu, P0 = g["X"], g["y"], g["mu"], g["P_lambda"]
    G, gv, _, _ = conjugate.regression_suffstats(X, y, None)
    s = {"beta": np.zeros((p, 1)), "tau": 1.0, "lambda": 0.01}
    draws = []
    for it in range(1500):
        s["beta"] = conjugate.normal_normal_dense_truncated(G, gv, s["tau"], P0, s["lambda"], mu, s["beta"], g["lower"],
                                                            g["upper"], rng.random(p))["x"]
        _, _, rss, cnt = conjugate.regression_suffstats(X, y, None, s["beta"])
        s["tau"], _, _ = conjugate.normal_gamma(1e-3, 1e-3, rss, cnt, rng.standard_gamma(1e-3 + cnt / 2))
        ss, cnt = conjugate.quadform(P0, s["beta"], mu)
        s["lambda"], _, _ = conjugate.normal_gamma(1e-3, 1e-3, ss, cnt, rng.standard_gamma(1e-3 + cnt / 2))
        if it >= 300:
            draws.append(s["beta"].ravel().copy())
    draws = np.array(draws)
    gpu_mean, cpu_mean = b.mean(axis=(0, 2)), draws.mean(axis=0)
    sd = draws.std(axis=0)
    assert np.all(np.abs(gpu_mean - cpu_mean) < 0.15 * sd + 5e-3), (gpu_mean, cpu_mean, sd)


@pytest.mark.parametrize("kind", [EYE, DENSE])
def test_sharding_invariance(kind):
    """64 chains with Philox uniforms against their second half launched alone with chain_offset = 32: bit-identical
    (the RNG is keyed by the global chain id, and a chain's scan does not depend on its neighbours)."""
    from openmcmc_b200 import kernels as K

    pr = _problem(64, 100, kind, False, seed=31)
    full, _, _, _ = _launch(pr, u=False, rng=K.rng(seed=8, site=2))
    half, _, _, _ = _launch(pr, u=False, rng=K.rng(seed=8, site=2, chain_offset=32), chains=slice(32, 64))
    np.testing.assert_array_equal(half, full[32:])
    assert not np.array_equal(full[0], full[1])


@pytest.mark.parametrize("kind", [EYE, DENSE])
def test_non_pd_chain_is_flagged_and_others_unchanged(kind):
    """A chain with Q_ii <= 0 (negative lambda) inside a batch gets OMC_STATUS_NOT_PD; every other chain's draw is
    the same, bit for bit, as in the batch without it (Philox uniforms)."""
    from openmcmc_b200 import kernels as K

    pr = _problem(40, 160, kind, False, seed=77)
    good, st_good, _, _ = _launch(pr, u=False, rng=K.rng(seed=9, site=4))
    lam = pr["lam"].copy()
    lam[17] = -50.0
    bad, st_bad, _, _ = _launch(pr, lam=lam, u=False, rng=K.rng(seed=9, site=4))
    assert not st_good.any()
    assert st_bad[17] & 1 and not np.delete(st_bad, 17).any()
    np.testing.assert_array_equal(np.delete(bad, 17, axis=0), np.delete(good, 17, axis=0))


def test_refuses_p_above_512():
    """p = 513: NotImplementedError from gmrf, PlanError from MCMC, before any launch."""
    from test_gpu_mcmc_regression import build

    from openmcmc_b200 import gmrf
    from openmcmc_b200.engine import PlanError
    from openmcmc_b200.mcmc import MCMC

    p = 513
    with pytest.raises(NotImplementedError, match="512"):
        gmrf.gibbs_canonical_truncated_normal(np.ones((p, 1)), np.eye(p), np.zeros((p, 1)), 0.0, 1.0,
                                              u=np.full(p, 0.5))
    g = _gdict(600, p, seed=5, lower=0.0)
    mdl, samplers, state = build(g)
    with pytest.raises(PlanError):
        MCMC(state, samplers, model=mdl, n_burn=0, n_iter=1).run_mcmc()
