"""GPU parity: the full MCMC driver on the Gibbs regression model (BASELINE configs[0] shape and friends) replays the
reference's golden chains when the reference's random streams are injected (debug_draws).  Tolerance 1e-9 on draws,
1e-10 on deterministic quantities (BASELINE.json north_star)."""

import glob
import os

import numpy as np
import pytest
from scipy import sparse

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
NAMES = sorted(os.path.basename(f)[:-4] for f in glob.glob(os.path.join(GOLD, "regression_*.npz")))


TRUNC_NAMES = sorted(os.path.basename(f)[:-4] for f in glob.glob(os.path.join(GOLD, "truncreg_*.npz")))


def build(g, n_chains=1, response=True):
    from openmcmc_b200.distribution.distribution import Gamma
    from openmcmc_b200.distribution.location_scale import Normal
    from openmcmc_b200.model import Model
    from openmcmc_b200.parameter import LinearCombination, ScaledMatrix
    from openmcmc_b200.sampler.sampler import NormalGamma, NormalNormal

    X, y, mu = g["X"], g["y"], g["mu"]
    n, p = X.shape
    P_tau = sparse.diags(g["w"], format="csc") if g["w"].size else sparse.csc_matrix(np.eye(n))
    P_lambda = g["P_lambda"]
    if str(g["prior"]) != "dense":
        P_lambda = sparse.csc_matrix(P_lambda)
    mdl = Model(
        [Normal("y", mean=LinearCombination(form={"beta": "X"}), precision=ScaledMatrix(matrix="P_tau", scalar="tau")),
         Normal("beta", mean="mu", precision=ScaledMatrix(matrix="P_lambda", scalar="lambda"),
                domain_response_lower=g["lower"].reshape(-1, 1) if "lower" in g and np.isfinite(g["lower"][0]) else None,
                domain_response_upper=g["upper"].reshape(-1, 1) if "upper" in g and np.isfinite(g["upper"][0]) else None),
         Gamma("tau", shape="a_tau", rate="b_tau"),
         Gamma("lambda", shape="a_lambda", rate="b_lambda")],
        response={"y": "mean"} if response else None,
    )
    smap = {"beta": NormalNormal("beta", mdl), "tau": NormalGamma("tau", mdl), "lambda": NormalGamma("lambda", mdl)}
    samplers = [smap[str(k)] for k in g["order"]]
    state = {"y": y, "X": X, "beta": np.zeros((p, 1)), "P_tau": P_tau, "tau": 1.0, "P_lambda": P_lambda, "mu": mu,
             "lambda": 0.01, "a_tau": 1e-3, "b_tau": 1e-3, "a_lambda": 1e-3, "b_lambda": 1e-3}
    return mdl, samplers, state


@pytest.mark.parametrize("name", NAMES)
def test_mcmc_replays_reference_chain(name):
    from openmcmc_b200.mcmc import MCMC
    from test_oracle_vs_golden import _load

    g = _load(name)
    mdl, samplers, state = build(g)
    n_iter = g["store_beta"].shape[1]
    dd = {"beta": {"z": g["z"]}, "tau": {"g": g["g_tau"]}, "lambda": {"g": g["g_lambda"]}}
    M = MCMC(state, samplers, model=mdl, n_burn=0, n_iter=n_iter, debug_draws=dd)
    M.run_mcmc()
    assert M.store["beta"].shape == g["store_beta"].shape
    assert M.store["tau"].shape == g["store_tau"].shape
    assert M.store["log_post"].shape == g["store_log_post"].shape
    np.testing.assert_allclose(M.store["beta"], g["store_beta"], rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(M.store["tau"], g["store_tau"], rtol=1e-9)
    np.testing.assert_allclose(M.store["lambda"], g["store_lambda"], rtol=1e-9)
    np.testing.assert_allclose(M.store["log_post"], g["store_log_post"], rtol=1e-10)
    np.testing.assert_allclose(M.store["y"], g["store_y"], rtol=1e-9, atol=1e-11)
    np.testing.assert_allclose(M.state["beta"], g["store_beta"][:, [-1]], rtol=1e-9, atol=1e-12)


@pytest.mark.parametrize("name", TRUNC_NAMES)
def test_mcmc_replays_truncated_reference_chain(name):
    """SURVEY §8 f3: truncated Normal prior -> coordinate-wise truncated Gibbs scan (sampler.py:196-205,
    gmrf.py:201-266), replayed with the reference's truncnorm.rvs uniforms."""
    from openmcmc_b200.mcmc import MCMC

    g = dict(np.load(os.path.join(GOLD, name + ".npz")))
    mdl, samplers, state = build(g)
    n_iter = g["store_beta"].shape[1]
    dd = {"beta": {"u": g["tn_u"]}, "tau": {"g": g["g_tau"]}, "lambda": {"g": g["g_lambda"]}}
    M = MCMC(state, samplers, model=mdl, n_burn=0, n_iter=n_iter, debug_draws=dd)
    M.run_mcmc()
    np.testing.assert_allclose(M.store["beta"], g["store_beta"], rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(M.store["tau"], g["store_tau"], rtol=1e-9)
    np.testing.assert_allclose(M.store["lambda"], g["store_lambda"], rtol=1e-9)
    np.testing.assert_allclose(M.store["log_post"], g["store_log_post"], rtol=1e-10)
    np.testing.assert_allclose(M.store["y"], g["store_y"], rtol=1e-9, atol=1e-11)


def test_truncated_free_running_stays_inside_and_matches_oracle_chain():
    """Free-running truncated Gibbs (Philox uniforms): every draw inside the bounds; per-coordinate posterior means
    agree with a free-running CPU oracle chain (numpy RNG) within Monte-Carlo error."""
    from openmcmc_b200.mcmc import MCMC
    from oracle import conjugate

    g = dict(np.load(os.path.join(GOLD, "truncreg_n120_p6_two_sided.npz")))
    mdl, samplers, state = build(g, response=False)
    C = 32
    M = MCMC(state, samplers, model=mdl, n_burn=100, n_iter=200, n_chains=C, seed=11)
    M.run_mcmc()
    b = M.store["beta"]                                      # (C, p, n_iter)
    lo, hi = g["lower"][0], g["upper"][0]
    assert np.all(b >= lo) and np.all(b <= hi)
    assert np.std(b[:, 0, -1]) > 0
    rng = np.random.default_rng(3)
    X, y, mu, P0 = g["X"], g["y"], g["mu"], g["P_lambda"]
    p = X.shape[1]
    G, gv, _, _ = conjugate.regression_suffstats(X, y, None)
    s = {"beta": np.zeros((p, 1)), "tau": 1.0, "lambda": 0.01}
    draws = []
    for it in range(2500):
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


def test_mcmc_replays_two_term_mean_chain():
    """y ~ N(X beta + Z gamma, .): every NormalNormal runs the fused pass on y minus the other term's predictor
    (omc_linear_predictor(residual_of=y), sampler.py:188-192); fitted values and log_post use both terms."""
    from openmcmc_b200.distribution.distribution import Gamma
    from openmcmc_b200.distribution.location_scale import Normal
    from openmcmc_b200.mcmc import MCMC
    from openmcmc_b200.model import Model
    from openmcmc_b200.parameter import LinearCombination, ScaledMatrix
    from openmcmc_b200.sampler.sampler import NormalGamma, NormalNormal

    g = dict(np.load(os.path.join(GOLD, "twoterm_n150_p7_q4.npz")))
    n, p, q = g["X"].shape[0], g["X"].shape[1], g["Z"].shape[1]
    mdl = Model(
        [Normal("y", mean=LinearCombination(form={"beta": "X", "gamma": "Z"}), precision=ScaledMatrix(matrix="W", scalar="tau")),
         Normal("beta", mean="mu_b", precision=ScaledMatrix(matrix="P_b", scalar="lam_b")),
         Normal("gamma", mean="mu_g", precision=ScaledMatrix(matrix="P_g", scalar="lam_g")),
         Gamma("tau", shape="a_tau", rate="b_tau"),
         Gamma("lam_b", shape="a_lam", rate="b_lam")],
        response={"y": "mean"})
    samplers = [NormalNormal("beta", mdl), NormalNormal("gamma", mdl), NormalGamma("tau", mdl), NormalGamma("lam_b", mdl)]
    state = {"y": g["y"], "X": g["X"], "Z": g["Z"], "W": sparse.diags(g["w"], format="csc"), "beta": np.zeros((p, 1)),
             "gamma": np.zeros((q, 1)), "tau": 1.0, "mu_b": g["mu_b"], "P_b": g["P_b"], "lam_b": 0.5,
             "mu_g": np.zeros((q, 1)), "P_g": sparse.identity(q, format="csc"), "lam_g": float(g["lam_g"]),
             "a_tau": 1e-3, "b_tau": 1e-3, "a_lam": 1.0, "b_lam": 1.0}
    dd = {"beta": {"z": g["z_beta"]}, "gamma": {"z": g["z_gamma"]}, "tau": {"g": g["g_tau"]}, "lam_b": {"g": g["g_lam"]}}
    C = 3
    dd_c = {k: {kk: np.repeat(np.asarray(vv)[:, None], C, axis=1) for kk, vv in v.items()} for k, v in dd.items()}
    M = MCMC(state, samplers, model=mdl, n_burn=0, n_iter=g["store_beta"].shape[1], n_chains=C, debug_draws=dd_c)
    M.run_mcmc()
    for c in range(C):
        np.testing.assert_allclose(M.store["beta"][c], g["store_beta"], rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(M.store["gamma"][c], g["store_gamma"], rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(M.store["tau"][c], g["store_tau"], rtol=1e-9)
        np.testing.assert_allclose(M.store["lam_b"][c], g["store_lam_b"], rtol=1e-9)
        np.testing.assert_allclose(M.store["y"][c], g["store_y"], rtol=1e-9, atol=1e-11)
    np.testing.assert_allclose(M.store["log_post"][:, 0], g["store_log_post"][:, 0], rtol=1e-10)


def test_mcmc_burn_thin_schedule_and_chains():
    """Iteration numbering (mcmc.py:97-103): (n_burn+n_iter)*n_thin sweeps; identical injected draws on every chain
    give identical chains; batched shapes (C, size, n_iter)."""
    from openmcmc_b200.mcmc import MCMC

    g = dict(np.load(os.path.join(GOLD, "regression_n50_p3.npz")))
    mdl, samplers, state = build(g, response=False)
    C = 5
    # 6 recorded sweeps = n_burn 2 + n_iter 2 with n_thin... use n_thin=1: burn 2, iter 4
    dd = {"beta": {"z": np.repeat(g["z"][:, None, :], C, axis=1)},
          "tau": {"g": np.repeat(g["g_tau"][:, None], C, axis=1)},
          "lambda": {"g": np.repeat(g["g_lambda"][:, None], C, axis=1)}}
    M = MCMC(state, samplers, model=mdl, n_burn=2, n_iter=4, n_chains=C, debug_draws=dd)
    M.run_mcmc()
    assert M.store["beta"].shape == (C, 3, 4)
    assert M.store["log_post"].shape == (4, C)
    for c in range(C):
        np.testing.assert_allclose(M.store["beta"][c], g["store_beta"][:, 2:], rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(M.store["tau"][c], g["store_tau"][:, 2:], rtol=1e-9)
    # thinning: n_thin=2, n_iter=3 stores sweeps 1,3,5
    M2 = MCMC(state, samplers, model=mdl, n_burn=0, n_iter=3, n_thin=2, n_chains=C, debug_draws=dd)
    M2.run_mcmc()
    np.testing.assert_allclose(M2.store["beta"][0], g["store_beta"][:, 1::2], rtol=1e-9, atol=1e-12)
    assert M2.launches_per_sweep() == 3      # draw (+ rss epilogue), fused {Gamma draws, quadratic form}, sweep counter


def test_mcmc_free_running_posterior_matches_truth():
    """Free-running chains (Philox): posterior mean of beta close to the least-squares solution; many chains agree
    within Monte-Carlo error; different chains differ; results independent of chain_offset sharding."""
    from openmcmc_b200.mcmc import MCMC

    g = dict(np.load(os.path.join(GOLD, "regression_n50_p3.npz")))
    mdl, samplers, state = build(g, response=False)
    C = 64
    M = MCMC(state, samplers, model=mdl, n_burn=200, n_iter=300, n_chains=C, seed=123)
    M.run_mcmc()
    b = M.store["beta"]                      # (C, 3, 300)
    ls = np.linalg.lstsq(g["X"], g["y"], rcond=None)[0].ravel()
    np.testing.assert_allclose(b.mean(axis=(0, 2)), ls, atol=0.02)
    assert np.std(b[:, 0, -1]) > 0
    tau_mean = M.store["tau"].mean()
    resid = g["y"] - g["X"] @ ls.reshape(-1, 1)
    assert abs(tau_mean - 1.0 / np.var(resid)) / tau_mean < 0.15
    # sharding invariance: chains 32..63 computed alone with chain_offset=32 reproduce the same draws
    M2 = MCMC(state, samplers, model=mdl, n_burn=200, n_iter=300, n_chains=32, seed=123, chain_offset=32)
    M2.run_mcmc()
    np.testing.assert_array_equal(M2.store["beta"], b[32:])


def test_sampler_single_call_reference_kats():
    """The reference's own known-answer tests for NormalNormal / NormalGamma (tests/test_sampler.py:262-341) through
    the same `.sample(state)` call, with its rvs patches expressed as debug_draws."""
    from openmcmc_b200 import parameter
    from openmcmc_b200.distribution.distribution import Gamma
    from openmcmc_b200.distribution.location_scale import Normal
    from openmcmc_b200.model import Model
    from openmcmc_b200.sampler.sampler import NormalGamma, NormalNormal

    for n, p in [(1, 1), (1, 10), (10, 1), (10, 10)]:
        rng = np.random.default_rng(0)
        state = {}
        state["prefactor_matrix"] = rng.random((n, p))
        state["parameter"] = rng.random((p, 1))
        state["response"] = state["prefactor_matrix"] @ state["parameter"]
        state["prior_mean"] = rng.random((1, 1)) * np.ones((p, 1))
        state["precision_matrix"] = np.diag(rng.random(n) + 0.1)
        state["prior_precision_vector"] = 0.1 + rng.random(1)
        state["prior_precision_matrix"] = np.eye(p)
        state["gamma_shape"] = 1e-3 * np.ones(1)
        state["gamma_rate"] = 1e-3 * np.ones(1)
        model = Model([
            Normal("response", mean=parameter.LinearCombination(form={"parameter": "prefactor_matrix"}),
                   precision=parameter.Identity("precision_matrix")),
            Normal("parameter", mean=parameter.Identity("prior_mean"),
                   precision=parameter.ScaledMatrix(matrix="prior_precision_matrix", scalar="prior_precision_vector")),
            Gamma("prior_precision_vector", shape=parameter.Identity("gamma_shape"), rate=parameter.Identity("gamma_rate")),
        ])
        nn = NormalNormal("parameter", model)
        # 1) X = 0 and z = 0 -> prior mean (test_sampler.py:274-277)
        ts = dict(state)
        ts["prefactor_matrix"] = np.zeros((n, p))
        out = nn.sample(dict(ts), debug_draws={"z": np.zeros(p)})
        np.testing.assert_allclose(out["parameter"], state["prior_mean"])
        # 2) prior precision 0, z = 0 -> weighted least squares (test_sampler.py:279-288); needs n >= p for full rank
        W = state["precision_matrix"]
        Xm = state["prefactor_matrix"]
        if n >= p and n > 1:
            ts = dict(state)
            ts["prior_precision_vector"] = np.zeros(1)
            out = nn.sample(dict(ts), debug_draws={"z": np.zeros(p)})
            np.testing.assert_allclose(out["parameter"], np.linalg.solve(Xm.T @ W @ Xm, Xm.T @ W @ state["response"]))
        # 3) zero means, z = 1 -> solve(chol(X'WX + Q0).T, 1) (test_sampler.py:290-308)
        ts = dict(state)
        ts["response"] = np.zeros((n, 1))
        ts["prior_mean"] = np.zeros((p, 1))
        out = nn.sample(dict(ts), debug_draws={"z": np.ones(p)})
        comp = np.linalg.solve(np.linalg.cholesky(Xm.T @ W @ Xm + state["prior_precision_vector"] * np.eye(p)).T,
                               np.ones((p, 1)))
        np.testing.assert_allclose(out["parameter"], comp)
        assert out["parameter"].shape == (p, 1)
        # NormalGamma: gamma.rvs -> a*scale, zero prior => 1/tau = mean(resid^2) (test_sampler.py:311-341)
        ng = NormalGamma("prior_precision_vector", model)
        ts = dict(state)
        ts["gamma_shape"] = np.zeros(1)
        ts["gamma_rate"] = np.zeros(1)
        out = ng.sample(dict(ts), debug_draws={"g": np.array([p / 2.0])})   # E[Gamma(a*,1)] = a* = p/2
        resid = ts["parameter"] - ts["prior_mean"]
        np.testing.assert_allclose(1 / out["prior_precision_vector"], np.mean(resid ** 2))
        # untouched keys (test_sampler.py:181-198)
        for k in ts:
            if k != "prior_precision_vector":
                np.testing.assert_allclose(out[k], ts[k])


def test_upload_blocks_give_identical_draws():
    """run_mcmc(upload_blocks=B): the chains run as B chain blocks whose uploads overlap the previous blocks' sweeps.
    Chains are independent and the RNG is keyed by the global chain id, so every stored draw, log_post, fitted value
    and final state equals the unblocked run bit for bit (ragged blocks included)."""
    import torch
    from scipy import sparse

    from openmcmc_b200.distribution.distribution import Gamma
    from openmcmc_b200.distribution.location_scale import Normal
    from openmcmc_b200.mcmc import MCMC
    from openmcmc_b200.model import Model
    from openmcmc_b200.parameter import LinearCombination, ScaledMatrix
    from openmcmc_b200.sampler.sampler import NormalGamma, NormalNormal

    rng = np.random.default_rng(5)
    C, n, p = 11, 300, 8
    X = rng.standard_normal((C, n, p))
    y = X @ rng.standard_normal((C, p, 1)) + 0.1 * rng.standard_normal((C, n, 1))
    mdl = Model([
        Normal("y", mean=LinearCombination(form={"beta": "X"}), precision=ScaledMatrix(matrix="P_tau", scalar="tau")),
        Normal("beta", mean="mu", precision=ScaledMatrix(matrix="P_lambda", scalar="lambda")),
        Gamma("tau", shape="a_tau", rate="b_tau"),
        Gamma("lambda", shape="a_lambda", rate="b_lambda")])
    mdl.response = {"y": "mean"}
    samplers = [NormalNormal("beta", mdl), NormalGamma("tau", mdl), NormalGamma("lambda", mdl)]

    def run(blocks, pinned):
        Xh = torch.as_tensor(X).pin_memory() if pinned else X
        state = {"y": y, "X": Xh, "beta": np.zeros((p, 1)), "P_tau": sparse.identity(n, format="csc"), "tau": 1.0,
                 "P_lambda": sparse.identity(p, format="csc"), "mu": np.zeros((p, 1)), "lambda": 0.01,
                 "a_tau": 1e-3, "b_tau": 1e-3, "a_lambda": 1e-3, "b_lambda": 1e-3}
        M = MCMC(state, samplers, model=mdl, n_burn=3, n_iter=5, n_thin=2, n_chains=C, seed=11, chain_offset=40,
                 upload_blocks=blocks)
        M.run_mcmc()
        return M

    A = run(1, False)
    for blocks, pinned in ((3, False), (4, True)):
        Bk = run(blocks, pinned)
        assert Bk.timing["upload_blocks"] == blocks
        assert set(Bk.store) == set(A.store)
        for key in A.store:
            assert Bk.store[key].shape == A.store[key].shape, key
            assert np.array_equal(Bk.store[key], A.store[key]), key
        for key in ("beta", "tau", "lambda"):
            assert np.array_equal(np.asarray(Bk.state[key]), np.asarray(A.state[key])), key
        assert np.array_equal(Bk.status, A.status)
    assert not np.array_equal(A.store["beta"][0], A.store["beta"][1])


def test_full_size_c2_properties():
    """BASELINE configs[1] at full size (4096 chains, n = 10,000, p = 64; 21 GB of X on the device): size-independent
    properties instead of an oracle run.  (a) the record of sampled chains against torch fp64 (G = X'X, g = X'y,
    rss(beta) of the fused pass and of the residual-only pass), (b) rss(beta = NULL) = y'y for every chain,
    (c) three free-running Gibbs sweeps of all chains equal, bit for bit, the same sweeps of a 1024-chain slice run on
    its own with chain_offset (chains are independent and the RNG is keyed by the global chain id; the slice is large
    enough for omc_reg_pass to pick the same row split, 592 chains or more -- with fewer chains per launch the rows
    are split over more CTAs and the sums agree to rounding instead)."""
    import torch
    from scipy import sparse

    from openmcmc_b200 import kernels as K
    from openmcmc_b200.distribution.distribution import Gamma
    from openmcmc_b200.distribution.location_scale import Normal
    from openmcmc_b200.mcmc import MCMC
    from openmcmc_b200.model import Model
    from openmcmc_b200.parameter import LinearCombination, ScaledMatrix
    from openmcmc_b200.sampler.sampler import NormalGamma, NormalNormal

    K.init_device(0)
    if torch.cuda.mem_get_info()[0] < 60e9:
        pytest.skip("needs 60 GB of free HBM")
    C, n, p = 4096, 10_000, 64
    gen = torch.Generator(device="cuda").manual_seed(2024)
    X = torch.randn(C, n, p, dtype=torch.float64, device="cuda", generator=gen)
    X[:, :, 0] = 1.0
    bt = torch.randn(C, p, 1, dtype=torch.float64, device="cuda", generator=gen)
    y = torch.bmm(X, bt) + 0.1 * torch.randn(C, n, 1, dtype=torch.float64, device="cuda", generator=gen)
    beta = torch.randn(C, p, dtype=torch.float64, device="cuda", generator=gen)
    rec = p * p + p + 2
    stats = torch.empty(C, rec, dtype=torch.float64, device="cuda")
    ns, ws = K.reg_pass_workspace(C, n, p)
    work = torch.empty(max(ws, 1), dtype=torch.float64, device="cuda")
    # (b) beta = NULL: rss = y'y
    K.reg_pass(X, y, None, None, stats, work, C, n, p)
    yy = (y[:, :, 0] ** 2).sum(dim=1)
    assert float(((stats[:, p * p + p] - yy).abs() / yy).max()) < 1e-12
    # (a) fused pass, then the residual-only pass with another beta
    K.reg_pass(X, y, None, beta, stats, work, C, n, p)
    first = stats.clone()
    beta2 = beta + 0.5
    K.reg_rss(X, y, None, beta2, stats, work, C, n, p)
    torch.cuda.synchronize()
    assert torch.equal(stats[:, : p * p + p], first[:, : p * p + p])
    for c in (0, 1, 777, 2048, 4095):
        G = X[c].T @ X[c]
        g = X[c].T @ y[c, :, 0]
        assert float((first[c, : p * p].reshape(p, p) - G).abs().max() / G.abs().max()) < 1e-12
        assert float((first[c, p * p : p * p + p] - g).abs().max() / g.abs().max()) < 1e-12
        for st, b in ((first, beta), (stats, beta2)):
            r = y[c, :, 0] - X[c] @ b[c]
            rss = float(r @ r)
            assert abs(float(st[c, p * p + p]) - rss) < 1e-11 * rss
        assert float(first[c, p * p + p + 1]) == n
    del stats, first, work
    # (c) sharding invariance of the whole Gibbs sweep at full size
    mdl = Model([
        Normal("y", mean=LinearCombination(form={"beta": "X"}), precision=ScaledMatrix(matrix="P_tau", scalar="tau")),
        Normal("beta", mean="mu", precision=ScaledMatrix(matrix="P_lambda", scalar="lambda")),
        Gamma("tau", shape="a_tau", rate="b_tau"),
        Gamma("lambda", shape="a_lambda", rate="b_lambda")])
    samplers = [NormalNormal("beta", mdl), NormalGamma("tau", mdl), NormalGamma("lambda", mdl)]

    def run(Xs, ys, nch, off):
        state = {"y": ys, "X": Xs, "beta": np.zeros((p, 1)), "P_tau": sparse.identity(n, format="csc"), "tau": 1.0,
                 "P_lambda": sparse.identity(p, format="csc"), "mu": np.zeros((p, 1)), "lambda": 0.01,
                 "a_tau": 1e-3, "b_tau": 1e-3, "a_lambda": 1e-3, "b_lambda": 1e-3}
        M = MCMC(state, samplers, model=mdl, n_burn=0, n_iter=3, n_chains=nch, seed=9, chain_offset=off)
        M.run_mcmc()
        return M

    full = run(X, y, C, 0)
    assert int((full.status != 0).sum()) == 0
    lo, hi = 1000, 2024
    part = run(X[lo:hi].contiguous(), y[lo:hi].contiguous(), hi - lo, lo)
    for key in ("beta", "tau", "lambda"):
        assert np.array_equal(full.store[key][lo:hi], part.store[key]), key
    assert np.array_equal(full.store["log_post"][:, lo:hi], part.store["log_post"])
    # the posterior mean of beta after 3 sweeps is already at the least-squares solution of its chain (noise sd 0.1)
    err = np.abs(full.store["beta"][:, :, -1] - bt[:, :, 0].cpu().numpy()).max()
    assert err < 0.05, err


MULTILIK = sorted(os.path.basename(f)[:-4] for f in glob.glob(os.path.join(GOLD, "multilik_*.npz")))


@pytest.mark.parametrize("name", MULTILIK)
def test_mcmc_replays_multi_likelihood_chain(name):
    """NormalNormal with several likelihood terms (sampler.py:179-192): two regressions on the same coefficients,
    optionally a direct observation (Identity mean, sampler.py:187-188), optionally a tridiagonal (GMRF) prior on the
    coefficients -- golden chains of the live reference, its variates injected."""
    from openmcmc_b200.distribution.distribution import Gamma
    from openmcmc_b200.distribution.location_scale import Normal
    from openmcmc_b200.mcmc import MCMC
    from openmcmc_b200.model import Model
    from openmcmc_b200.parameter import LinearCombination, ScaledMatrix
    from openmcmc_b200.sampler.sampler import NormalGamma, NormalNormal

    g = dict(np.load(os.path.join(GOLD, name + ".npz")))
    n1, p = g["X1"].shape
    n2 = g["X2"].shape[0]
    names = [str(k) for k in g["names"]]
    P_lambda = sparse.csc_matrix(g["P_lambda"])
    dists = [Normal("y1", mean=LinearCombination(form={"beta": "X1"}), precision=ScaledMatrix(matrix="P1", scalar="tau1")),
             Normal("y2", mean=LinearCombination(form={"beta": "X2"}), precision=ScaledMatrix(matrix="P2", scalar="tau2")),
             Normal("beta", mean="mu", precision=ScaledMatrix(matrix="P_lambda", scalar="lambda")),
             Gamma("tau1", shape="a", rate="b"), Gamma("tau2", shape="a", rate="b"), Gamma("lambda", shape="a", rate="b")]
    state = {"y1": g["y1"], "y2": g["y2"], "X1": g["X1"], "X2": g["X2"], "beta": np.zeros((p, 1)),
             "P1": sparse.identity(n1, format="csc"), "P2": sparse.diags(g["w2"], format="csc"), "tau1": 1.0, "tau2": 1.0,
             "P_lambda": P_lambda, "mu": np.zeros((p, 1)), "lambda": 0.1, "a": 1e-3, "b": 1e-3}
    if bool(g["identity_term"]):
        dists.insert(2, Normal("y3", mean="beta", precision=ScaledMatrix(matrix="P3", scalar="tau3")))
        dists.append(Gamma("tau3", shape="a", rate="b"))
        state.update({"y3": g["y3"], "P3": sparse.identity(p, format="csc"), "tau3": 1.0})
    mdl = Model(dists)
    samplers = [NormalNormal("beta", mdl)] + [NormalGamma(k, mdl) for k in names[1:]]
    n_iter = g["store_beta"].shape[1]
    dd = {"beta": {"z": g["z"]}}
    dd.update({k: {"g": g["g_" + k]} for k in names[1:]})
    M = MCMC(state, samplers, model=mdl, n_burn=0, n_iter=n_iter, debug_draws=dd)
    M.run_mcmc()
    np.testing.assert_allclose(M.store["beta"], g["store_beta"], rtol=1e-9, atol=1e-12)
    for k in names[1:]:
        np.testing.assert_allclose(M.store[k], g["store_" + k], rtol=1e-9)
    np.testing.assert_allclose(M.store["log_post"], g["store_log_post"], rtol=1e-10)


def test_scaled_matrix_predictor_and_parameter_grads():
    """ScaledMatrix.predictor (parameter.py:319-329) and Parameter.grad (parameter.py:125-141, 218-228, 282-297, 349-360)."""
    from openmcmc_b200.parameter import Identity, LinearCombination, LinearCombinationWithTransform, ScaledMatrix

    rng = np.random.default_rng(0)
    P = sparse.diags([rng.random(6) + 1.0, -rng.random(5)], [0, 1], format="csc")
    state = {"P": P, "tau": np.array([[2.5]]), "D": rng.standard_normal((4, 4)), "X": rng.standard_normal((5, 3)),
             "b": rng.standard_normal((3, 1))}
    sm = ScaledMatrix(matrix="P", scalar="tau")
    out = sm.predictor(state)
    assert sparse.issparse(out) and np.allclose(out.toarray(), 2.5 * P.toarray(), rtol=1e-15)
    np.testing.assert_allclose(ScaledMatrix(matrix="D", scalar="tau").predictor(state), 2.5 * state["D"], rtol=1e-15)
    assert sm.grad(state, "tau") is state["P"]
    assert np.array_equal(Identity("b").grad(state, "b"), np.eye(3)) and not Identity("b").grad(state, "x").any()
    assert np.array_equal(LinearCombination({"b": "X"}).grad(state, "b"), state["X"].T)
    lt = LinearCombinationWithTransform(form={"b": "X"}, transform={"b": True})
    np.testing.assert_allclose(lt.grad(state, "b"), np.exp(state["b"]) * state["X"].T, rtol=1e-14)
    with pytest.raises(ValueError):
        ScaledMatrix(matrix="D", scalar="D").predictor(state)
