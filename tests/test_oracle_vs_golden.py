"""CPU: the numpy oracle reproduces the reference's golden vectors (tests/golden/*.npz, made by make_golden.py from
the live reference with injected random streams).  This is what pins the oracle."""

import glob
import hashlib
import os

import numpy as np
import pytest

from oracle import conjugate, dist, gmrf

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _load(name):
    """A golden case.  A design matrix too large to store (n700_p200: 1.1 MB of float64) is kept as the seed that
    generated it (make_golden.regression_case) and the SHA-256 of its bytes; it is regenerated here and checked."""
    g = dict(np.load(os.path.join(GOLD, name + ".npz"), allow_pickle=False))
    if "X_seed" in g:
        X = np.random.default_rng(int(g["X_seed"])).standard_normal(tuple(g["X_shape"]))
        X[:, 0] = 1.0
        assert hashlib.sha256(X.tobytes()).hexdigest() == str(g["X_sha256"]), f"{name}: regenerated X differs"
        g["X"] = X
    return g


@pytest.mark.parametrize("name", sorted(os.path.basename(f)[:-4] for f in glob.glob(os.path.join(GOLD, "regression_*.npz"))))
def test_regression_chain_replay(name):
    g = _load(name)
    X, y, mu = g["X"], g["y"], g["mu"]
    n, p = X.shape
    w = g["w"] if g["w"].size else None
    P0 = g["P_lambda"]
    order = tuple(str(s) for s in g["order"])
    state = {"beta": np.zeros((p, 1)), "tau": 1.0, "lambda": 0.01, "a_tau": 1e-3, "b_tau": 1e-3, "a_lambda": 1e-3,
             "b_lambda": 1e-3}
    n_iter = g["store_beta"].shape[1]
    logdet_P0 = 2 * np.sum(np.log(np.diag(np.linalg.cholesky(P0))))
    logdet_W = 0.0 if w is None else float(np.sum(np.log(w)))
    for it in range(n_iter):
        state = conjugate.gibbs_regression_sweep(X, y, state, g["z"][it], g["g_tau"][it], g["g_lambda"][it], P0=P0,
                                                 mu0=mu, w=w, order=order)
        np.testing.assert_allclose(state["beta"].ravel(), g["store_beta"][:, it], rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(state["tau"], g["store_tau"][0, it], rtol=1e-10)
        np.testing.assert_allclose(state["lambda"], g["store_lambda"][0, it], rtol=1e-10)
        np.testing.assert_allclose((X @ state["beta"]).ravel(), g["store_y"][:, it], rtol=1e-9, atol=1e-11)
        _, _, rss, _ = conjugate.regression_suffstats(X, y, w, state["beta"])
        ssb, _ = conjugate.quadform(P0, state["beta"], mu)
        lp = (dist.normal_log_p_from_ss(n, state["tau"], logdet_W, rss)
              + dist.normal_log_p_from_ss(p, state["lambda"], logdet_P0, ssb)
              + dist.gamma_log_p(state["tau"], 1e-3, 1e-3) + dist.gamma_log_p(state["lambda"], 1e-3, 1e-3))
        np.testing.assert_allclose(lp, g["store_log_post"][it, 0], rtol=1e-10)


@pytest.mark.parametrize("name", sorted(os.path.basename(f)[:-4] for f in glob.glob(os.path.join(GOLD, "truncreg_*.npz"))))
def test_truncated_regression_chain_replay(name):
    """Truncated Normal prior on beta: NormalNormal.sample is one coordinate-wise truncated Gibbs scan
    (sampler.py:196-205, gmrf.py:201-266); replay of the reference chain with its truncnorm.rvs uniforms injected."""
    g = _load(name)
    X, y, mu = g["X"], g["y"], g["mu"]
    n, p = X.shape
    w = g["w"] if g["w"].size else None
    P0 = g["P_lambda"]
    state = {"beta": np.zeros((p, 1)), "tau": 1.0, "lambda": 0.01}
    if p == 1:
        assert g["lower"][0] > 0   # the start value 0 lies outside: the p == 1 branch ignores it (gmrf.py:245-248)
    for it in range(g["store_beta"].shape[1]):
        G, gv, _, _ = conjugate.regression_suffstats(X, y, w)
        state["beta"] = conjugate.normal_normal_dense_truncated(G, gv, state["tau"], P0, state["lambda"], mu,
                                                                state["beta"], g["lower"], g["upper"], g["tn_u"][it])["x"]
        np.testing.assert_allclose(state["beta"].ravel(), g["store_beta"][:, it], rtol=1e-9, atol=1e-12)
        assert np.all(state["beta"] >= g["lower"][0]) and np.all(state["beta"] <= g["upper"][0])
        _, _, rss, cnt = conjugate.regression_suffstats(X, y, w, state["beta"])
        state["tau"], _, _ = conjugate.normal_gamma(1e-3, 1e-3, rss, cnt, g["g_tau"][it])
        ss, cnt = conjugate.quadform(P0, state["beta"], mu)
        state["lambda"], _, _ = conjugate.normal_gamma(1e-3, 1e-3, ss, cnt, g["g_lambda"][it])
        np.testing.assert_allclose(state["tau"], g["store_tau"][0, it], rtol=1e-10)
        np.testing.assert_allclose(state["lambda"], g["store_lambda"][0, it], rtol=1e-10)


@pytest.mark.parametrize("name", sorted(os.path.basename(f)[:-4] for f in glob.glob(os.path.join(GOLD, "mixture_*.npz"))))
def test_mixture_chain_replay(name):
    """SURVEY f2: NormalNormal with a mixture prior, the NormalGamma K-loop and MixtureAllocation replay the reference
    chain (sampler.py:154-207, 272-288, 292-355) with its norm / gamma / uniform draws injected."""
    g = _load(name)
    X, y, w, prob = g["X"], g["y"], g["w"], g["prob"]
    n = X.shape[0]
    s = {"beta": g["beta0"], "mu": g["mu0"], "tau": g["tau0"], "z": g["z0"]}
    for it in range(g["store_beta"].shape[1]):
        s = conjugate.gibbs_mixture_sweep(X, y, w, s, prob, g["a_tau"], g["b_tau"], g["z_beta"][it], g["g"][it], g["u"][it])
        np.testing.assert_allclose(s["beta"].ravel(), g["store_beta"][:, it], rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(np.ravel(s["tau"]), g["store_tau"][:, it], rtol=1e-10)
        np.testing.assert_array_equal(np.ravel(s["z"]), g["store_z"][:, it])
        _, _, rss, _ = conjugate.regression_suffstats(X, y, w, s["beta"])
        lp = (dist.normal_log_p_from_ss(n, 1.0, float(np.sum(np.log(w))), rss)
              + conjugate.mixture_normal_log_p(s["beta"], s["mu"], s["tau"], s["z"])
              + dist.gamma_log_p(np.ravel(s["tau"]), np.ravel(g["a_tau"]), np.ravel(g["b_tau"]))
              + conjugate.categorical_log_p(s["z"], prob))
        np.testing.assert_allclose(lp, g["store_log_post"][it, 0], rtol=1e-10)


def test_two_term_regression_chain_replay():
    """Mean with two LinearCombination terms: each NormalNormal conditions on y minus the other term's predictor
    (sampler.py:188-192); NormalGamma(tau) uses the full residual (sampler.py:275-276)."""
    g = _load("twoterm_n150_p7_q4")
    X, Z, y, w = g["X"], g["Z"], g["y"], g["w"]
    n, p, q = X.shape[0], X.shape[1], Z.shape[1]
    beta, gamma, tau, lam_b = np.zeros((p, 1)), np.zeros((q, 1)), 1.0, 0.5
    for it in range(g["store_beta"].shape[1]):
        G, gv, _, _ = conjugate.regression_suffstats(X, y - Z @ gamma, w)
        beta = conjugate.normal_normal_dense(G, gv, tau, g["P_b"], lam_b, g["mu_b"], g["z_beta"][it])["x"]
        G, gv, _, _ = conjugate.regression_suffstats(Z, y - X @ beta, w)
        gamma = conjugate.normal_normal_dense(G, gv, tau, 1.0, float(g["lam_g"]), None, g["z_gamma"][it])["x"]
        _, _, rss, cnt = conjugate.regression_suffstats(X, y - Z @ gamma, w, beta)
        tau, _, _ = conjugate.normal_gamma(1e-3, 1e-3, rss, cnt, g["g_tau"][it])
        ss, cnt = conjugate.quadform(g["P_b"], beta, g["mu_b"])
        lam_b, _, _ = conjugate.normal_gamma(1.0, 1.0, ss, cnt, g["g_lam"][it])
        np.testing.assert_allclose(beta.ravel(), g["store_beta"][:, it], rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(gamma.ravel(), g["store_gamma"][:, it], rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(tau, g["store_tau"][0, it], rtol=1e-10)
        np.testing.assert_allclose(lam_b, g["store_lam_b"][0, it], rtol=1e-10)
        np.testing.assert_allclose((X @ beta + Z @ gamma).ravel(), g["store_y"][:, it], rtol=1e-9, atol=1e-11)


def test_truncnorm_restatement_matches_scipy():
    """oracle.gmrf truncated-normal helpers == scipy.stats.truncnorm (what gmrf.py:269-318 calls)."""
    from scipy import stats

    rng = np.random.default_rng(0)
    for _ in range(200):
        mean, scale = rng.normal() * 3, rng.random() * 2 + 0.05
        lo = mean + scale * rng.normal() * 3
        hi = lo + rng.random() * 5 * scale + 1e-3
        if rng.random() < 0.3:
            hi = np.inf
        if rng.random() < 0.2:
            lo = -np.inf
        u = rng.random()
        a, b = (lo - mean) / scale, (hi - mean) / scale
        x_ref = stats.truncnorm.ppf(u, a, b, loc=mean, scale=scale)
        x = gmrf.truncated_normal_rv(mean, scale, lo, hi, u)
        np.testing.assert_allclose(x, x_ref, rtol=1e-12, atol=1e-12)
        lp_ref = stats.truncnorm.logpdf(x_ref, a, b, loc=mean, scale=scale)
        lp = gmrf.truncated_normal_log_pdf(x_ref, mean, scale, lo, hi)
        np.testing.assert_allclose(lp, lp_ref, rtol=1e-11, atol=1e-11)
    assert gmrf.truncated_normal_log_pdf(-1.0, 0.0, 1.0, 0.0, np.inf) == -np.inf


def test_tridiag_restatement_matches_dense():
    """Thomas-order tridiagonal Cholesky == dense Cholesky of the same matrix (gmrf.py:489-520 contract)."""
    rng = np.random.default_rng(1)
    s = np.cumsum(rng.exponential(size=40))
    d, e = gmrf.precision_irregular_diagonals(s)
    d = 3.0 * d + 0.7
    e = 3.0 * e
    Q = np.diag(d) + np.diag(e, 1) + np.diag(e, -1)
    L = np.linalg.cholesky(Q)
    l, c = gmrf.tridiag_cholesky(d, e)
    np.testing.assert_allclose(l, np.diag(L), rtol=1e-13)
    np.testing.assert_allclose(c, np.diag(L, -1), rtol=1e-12)
    b, z = rng.normal(size=40), rng.normal(size=40)
    x, mu, _, _ = gmrf.tridiag_sample_canonical(d, e, b, z)
    x_ref, mu_ref, _ = gmrf.sample_normal_canonical(b.reshape(-1, 1), Q, z.reshape(-1, 1))
    np.testing.assert_allclose(mu, mu_ref.ravel(), rtol=1e-11)
    np.testing.assert_allclose(x, x_ref.ravel(), rtol=1e-11)
    np.testing.assert_allclose(gmrf.tridiag_quadform(d, e, z), z @ Q @ z, rtol=1e-12)
    np.testing.assert_allclose(gmrf.tridiag_logdet(d, e), np.linalg.slogdet(Q)[1], rtol=1e-12)


@pytest.mark.parametrize("name", sorted(os.path.basename(f)[:-4] for f in glob.glob(os.path.join(GOLD, "gmrf_*.npz"))))
def test_gmrf_chain_replay(name):
    """The tridiagonal restatement replays the reference's example-4 chains: the notebook form (dense LAPACK in the
    reference, SURVEY F4) and the sparse form (SuperLU, natural order).  Tolerance = kappa * eps scale (SURVEY B.6)."""
    g = _load(name)
    order = tuple(str(s) for s in g["order"])
    s = {"b": g["y"].copy(), "lambda": 100.0, "tau": 1.0, "a_lam": 10.0, "b_lam": 1.0, "a_tau": 1.0, "b_tau": 1.0}
    for it in range(g["store_b"].shape[1]):
        s = conjugate.gibbs_gmrf_sweep(g["pd"], g["pe"], g["w"], g["y"], g["mu"], s, g["z"][it], g["g_lambda"][it],
                                       g["g_tau"][it], order)
        np.testing.assert_allclose(s["b"], g["store_b"][:, it], rtol=1e-9, atol=1e-9)
        np.testing.assert_allclose(s["lambda"], g["store_lambda"][0, it], rtol=1e-9)
        np.testing.assert_allclose(s["tau"], g["store_tau"][0, it], rtol=1e-9)
        np.testing.assert_allclose(conjugate.gmrf_log_post(g["pd"], g["pe"], g["w"], g["y"], g["mu"], s),
                                   g["store_log_post"][it, 0], rtol=1e-10)


MULTILIK = sorted(os.path.basename(f)[:-4] for f in glob.glob(os.path.join(GOLD, "multilik_*.npz")))


def multilik_terms(g):
    p = g["X1"].shape[1]
    terms = [(g["X1"], g["y1"], None), (g["X2"], g["y2"], g["w2"])]
    if bool(g["identity_term"]):
        terms.append((np.eye(p), g["y3"], None))
    return terms


@pytest.mark.parametrize("name", MULTILIK)
def test_multi_likelihood_normal_normal_chain(name):
    """sampler.py:179-192: several likelihood terms (two regressions, optionally an Identity-mean observation of the
    coefficients, optionally a tridiagonal prior) -- the oracle sweep against the live reference's chain."""
    g = dict(np.load(os.path.join(GOLD, name + ".npz")))
    terms = multilik_terms(g)
    p = g["X1"].shape[1]
    names = [str(k) for k in g["names"]]
    st = {"beta": np.zeros((p, 1)), "taus": [1.0] * len(terms), "lam": 0.1}
    for it in range(g["store_beta"].shape[1]):
        gam = [g["g_" + k][it] for k in names[1:]]
        st = conjugate.multi_likelihood_sweep(terms, st, g["P_lambda"], np.zeros((p, 1)), g["z"][it], gam)
        np.testing.assert_allclose(st["beta"].ravel(), g["store_beta"][:, it], rtol=1e-9, atol=1e-12)
        for k, v in zip(names[1:-1], st["taus"]):
            np.testing.assert_allclose(v, g["store_" + k][0, it], rtol=1e-9)
        np.testing.assert_allclose(st["lam"], g["store_lambda"][0, it], rtol=1e-9)
