"""Generate golden vectors from the LIVE, unmodified reference (run in the build container only).

    python tests/golden/make_golden.py            # writes tests/golden/*.npz

The reference (/root/reference/src/openmcmc) is imported as-is; its random streams are replaced by recorded ones the
same way its own tests do it (monkeypatching scipy.stats.*.rvs, tests/test_sampler.py:211-215), so the very same
numbers can be injected into the oracle and into the CUDA kernels (debug_draws).  Nothing here runs on the GPU box:
the .npz files are committed.
"""

import hashlib
import os
import sys

import numpy as np
from scipy import sparse, stats

REF = "/root/reference/src"
sys.path.insert(0, REF)
OUT = os.path.dirname(os.path.abspath(__file__))

from openmcmc import gmrf  # noqa: E402
from openmcmc.distribution.distribution import Categorical, Gamma, Poisson, Uniform  # noqa: E402
from openmcmc.distribution.location_scale import LogNormal, Normal  # noqa: E402
from openmcmc.parameter import LinearCombinationWithTransform  # noqa: E402
from openmcmc.mcmc import MCMC  # noqa: E402
from openmcmc.model import Model  # noqa: E402
from openmcmc.parameter import Identity, LinearCombination, ScaledMatrix  # noqa: E402
from openmcmc.sampler.metropolis_hastings import ManifoldMALA, RandomWalk, RandomWalkLoop  # noqa: E402
from openmcmc.sampler.sampler import MixtureAllocation, NormalGamma, NormalNormal  # noqa: E402
from openmcmc.sampler.reversible_jump import ReversibleJump  # noqa: E402
from openmcmc.distribution.location_scale import NullDistribution  # noqa: E402
from openmcmc.parameter import MixtureParameterMatrix, MixtureParameterVector  # noqa: E402


class Streams:
    """Replay/record wrapper for the scipy.stats rvs entry points the reference uses (SURVEY F7)."""

    def __init__(self, seed):
        self.rng = np.random.default_rng(seed)
        self.log = {"z": [], "g": [], "u": [], "tn_u": [], "randint": []}
        self._saved = {}

    def norm_rvs(self, size=1, scale=1, loc=0):
        z = self.rng.standard_normal(size)
        self.log["z"].append(np.array(z, dtype=float).ravel())
        return loc + scale * z

    def gamma_rvs(self, a, scale=1, size=None):
        a = np.asarray(a, dtype=float)
        shp = np.broadcast(a, np.asarray(scale)).shape if size is None else size
        g = self.rng.standard_gamma(np.broadcast_to(a, shp))
        self.log["g"].append(np.array(g, dtype=float).ravel())
        return g * scale

    def uniform_rvs(self, size=None, loc=0, scale=1):
        u = self.rng.random(size)
        self.log["u"].append(np.array(u, dtype=float).ravel())
        return loc + scale * u

    def truncnorm_rvs(self, a, b, loc=0, scale=1, size=1):
        u = self.rng.random(size)
        self.log["tn_u"].append(np.array(u, dtype=float).ravel())
        return stats.truncnorm.ppf(u, a, b, loc=loc, scale=scale)

    def randint_rvs(self, low, high, size=None):
        k = int(self.rng.integers(int(np.asarray(low).ravel()[0]), int(np.asarray(high).ravel()[0])))
        self.log["randint"].append(np.array([k], dtype=float))
        return k

    def __enter__(self):
        for dist, name, fn in ((stats.norm, "rvs", self.norm_rvs), (stats.gamma, "rvs", self.gamma_rvs),
                               (stats.uniform, "rvs", self.uniform_rvs), (stats.truncnorm, "rvs", self.truncnorm_rvs),
                               (stats.randint, "rvs", self.randint_rvs)):
            self._saved[(dist, name)] = getattr(dist, name)
            setattr(dist, name, fn)
        return self

    def __exit__(self, *exc):
        for (dist, name), fn in self._saved.items():
            setattr(dist, name, fn)

    def stack(self, key):
        return np.array(self.log[key]) if self.log[key] else np.zeros((0,))


# ----------------------------------------------------------------------------------------------- regression (C1 shape)
def regression_case(n, p, seed, n_iter, weighted=False, order=("beta", "tau", "lambda"), prior="eye", trunc=None,
                    noise=0.1):
    """trunc = (lower, upper) (size-1 arrays or None): truncated Normal prior on beta -> NormalNormal.sample runs
    gmrf.gibbs_canonical_truncated_normal (sampler.py:196-205); its truncnorm.rvs uniforms are recorded in `tn_u`."""
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, p))
    X[:, 0] = 1.0
    beta_true = rng.standard_normal((p, 1))
    y = X @ beta_true + noise * rng.standard_normal((n, 1))
    if weighted:
        w = rng.random(n) + 0.2  # strictly positive: a singular P_tau breaks the reference's own log_p
        P_tau = sparse.diags(w, format="csc")
    else:
        P_tau = sparse.csc_matrix(np.eye(n))
    if prior == "eye":
        P_lambda = sparse.csc_matrix(np.eye(p))
    elif prior == "diag":
        P_lambda = sparse.diags(rng.random(p) + 0.5, format="csc")
    else:
        A = rng.standard_normal((p, p))
        P_lambda = A @ A.T + p * np.eye(p)
    mu = rng.standard_normal((p, 1)) * 0.1
    mdl = Model(
        [Normal("y", mean=LinearCombination(form={"beta": "X"}), precision=ScaledMatrix(matrix="P_tau", scalar="tau")),
         Normal("beta", mean="mu", precision=ScaledMatrix(matrix="P_lambda", scalar="lambda"),
                domain_response_lower=None if trunc is None else trunc[0],
                domain_response_upper=None if trunc is None else trunc[1]),
         Gamma("tau", shape="a_tau", rate="b_tau"),
         Gamma("lambda", shape="a_lambda", rate="b_lambda")],
        response={"y": "mean"},
    )
    smap = {"beta": NormalNormal("beta", mdl), "tau": NormalGamma("tau", mdl), "lambda": NormalGamma("lambda", mdl)}
    samplers = [smap[k] for k in order]
    state = {"y": y, "X": X, "beta": np.zeros((p, 1)), "P_tau": P_tau, "tau": 1.0, "P_lambda": P_lambda, "mu": mu,
             "lambda": 0.01, "a_tau": 1e-3, "b_tau": 1e-3, "a_lambda": 1e-3, "b_lambda": 1e-3}
    with Streams(seed + 1) as s:
        import openmcmc.mcmc as m

        m.tqdm = lambda it: it
        M = MCMC(state, samplers, model=mdl, n_burn=0, n_iter=n_iter)
        M.run_mcmc()
    z = s.stack("z")                      # [n_iter, p]
    g = s.stack("g")                      # [2*n_iter, 1] in sampler order (tau/lambda interleaved as in `order`)
    gorder = [k for k in order if k != "beta"]
    out = {
        "X": X, "y": y, "mu": mu, "w": (np.asarray(P_tau.diagonal()) if weighted else np.zeros(0)),
        "P_lambda": (P_lambda.toarray() if sparse.issparse(P_lambda) else P_lambda),
        "order": np.array(order), "z": z, "weighted": weighted, "prior": prior,
        "g_" + gorder[0]: g[0::2, 0], "g_" + gorder[1]: g[1::2, 0],
        "store_beta": M.store["beta"], "store_tau": M.store["tau"], "store_lambda": M.store["lambda"],
        "store_log_post": M.store["log_post"], "store_y": M.store["y"],
    }
    if trunc is not None:
        out["tn_u"] = s.stack("tn_u").reshape(n_iter, p)
        out["lower"] = np.array([-np.inf]) if trunc[0] is None else np.asarray(trunc[0], dtype=float).ravel()
        out["upper"] = np.array([np.inf]) if trunc[1] is None else np.asarray(trunc[1], dtype=float).ravel()
    if X.nbytes > 1 << 20:
        # random float64 does not compress: a design matrix over 1 MB is stored as its seed and digest instead, and
        # tests/test_oracle_vs_golden.py:_load regenerates it
        del out["X"]
        out.update(X_seed=np.array(seed), X_shape=np.array(X.shape),
                   X_sha256=np.array(hashlib.sha256(X.tobytes()).hexdigest()))
    return out


def regression_two_term_case(n, p, q, seed, n_iter):
    """Mean with two terms, y ~ N(X beta + Z gamma, (tau W)^-1): each NormalNormal works on y minus the other term
    (predictor_conditional(term_to_exclude), sampler.py:188-192); NormalGamma(tau) sees the full residual."""
    rng = np.random.default_rng(seed)
    X, Z = rng.standard_normal((n, p)), rng.standard_normal((n, q))
    y = X @ rng.standard_normal((p, 1)) + Z @ (0.5 * rng.standard_normal((q, 1))) + 0.3 * rng.standard_normal((n, 1))
    W = sparse.diags(rng.random(n) + 0.5, format="csc")
    A = rng.standard_normal((p, p))
    P_b = A @ A.T / p + np.eye(p)
    mdl = Model(
        [Normal("y", mean=LinearCombination(form={"beta": "X", "gamma": "Z"}), precision=ScaledMatrix(matrix="W", scalar="tau")),
         Normal("beta", mean="mu_b", precision=ScaledMatrix(matrix="P_b", scalar="lam_b")),
         Normal("gamma", mean="mu_g", precision=ScaledMatrix(matrix="P_g", scalar="lam_g")),
         Gamma("tau", shape="a_tau", rate="b_tau"),
         Gamma("lam_b", shape="a_lam", rate="b_lam")],
        response={"y": "mean"},
    )
    samplers = [NormalNormal("beta", mdl), NormalNormal("gamma", mdl), NormalGamma("tau", mdl), NormalGamma("lam_b", mdl)]
    state = {"y": y, "X": X, "Z": Z, "W": W, "beta": np.zeros((p, 1)), "gamma": np.zeros((q, 1)), "tau": 1.0,
             "mu_b": 0.1 * rng.standard_normal((p, 1)), "P_b": P_b, "lam_b": 0.5, "mu_g": np.zeros((q, 1)),
             "P_g": sparse.identity(q, format="csc"), "lam_g": 2.0, "a_tau": 1e-3, "b_tau": 1e-3, "a_lam": 1.0, "b_lam": 1.0}
    mu_b = state["mu_b"].copy()
    with Streams(seed + 1) as s:
        M = _run_ref(state, samplers, mdl, n_iter)
    zs = s.log["z"]
    g = s.stack("g")
    return {"X": X, "Z": Z, "y": y, "w": np.asarray(W.diagonal()), "P_b": P_b, "mu_b": mu_b, "lam_g": 2.0,
            "z_beta": np.array(zs[0::2]), "z_gamma": np.array(zs[1::2]), "g_tau": g[0::2, 0], "g_lam": g[1::2, 0],
            "store_beta": M.store["beta"], "store_gamma": M.store["gamma"], "store_tau": M.store["tau"],
            "store_lam_b": M.store["lam_b"], "store_log_post": M.store["log_post"], "store_y": M.store["y"]}


# ----------------------------------------------------------------------------------------------- Metropolis-Hastings (C4 shape)
def multilik_case(n1, n2, p, seed, n_iter, identity_term=True, gmrf_prior=False):
    """NormalNormal with SEVERAL likelihood terms (sampler.py:179-192): two regressions on the same coefficients, and
    optionally a direct noisy observation of the coefficients (Identity mean, sampler.py:187-188); with gmrf_prior the
    prior precision is the tridiagonal RW1 matrix (example 4's prior on regression coefficients)."""
    rng = np.random.default_rng(seed)
    X1, X2 = rng.standard_normal((n1, p)), rng.standard_normal((n2, p))
    beta_true = np.cumsum(rng.standard_normal((p, 1)) * 0.3, axis=0) if gmrf_prior else rng.standard_normal((p, 1))
    y1 = X1 @ beta_true + 0.1 * rng.standard_normal((n1, 1))
    y2 = X2 @ beta_true + 0.3 * rng.standard_normal((n2, 1))
    y3 = beta_true + 0.5 * rng.standard_normal((p, 1))
    w2 = rng.random(n2) + 0.3
    if gmrf_prior:
        P_lambda = gmrf.precision_irregular(np.cumsum(rng.exponential(size=p) + 0.5)).tolil()
        P_lambda[0, 0] += 0.1
        P_lambda = P_lambda.tocsc()
    else:
        P_lambda = sparse.csc_matrix(np.eye(p))
    dists = [Normal("y1", mean=LinearCombination(form={"beta": "X1"}), precision=ScaledMatrix(matrix="P1", scalar="tau1")),
             Normal("y2", mean=LinearCombination(form={"beta": "X2"}), precision=ScaledMatrix(matrix="P2", scalar="tau2")),
             Normal("beta", mean="mu", precision=ScaledMatrix(matrix="P_lambda", scalar="lambda")),
             Gamma("tau1", shape="a", rate="b"), Gamma("tau2", shape="a", rate="b"), Gamma("lambda", shape="a", rate="b")]
    state = {"y1": y1, "y2": y2, "X1": X1, "X2": X2, "beta": np.zeros((p, 1)), "P1": sparse.identity(n1, format="csc"),
             "P2": sparse.diags(w2, format="csc"), "tau1": 1.0, "tau2": 1.0, "P_lambda": P_lambda, "mu": np.zeros((p, 1)),
             "lambda": 0.1, "a": 1e-3, "b": 1e-3}
    names = ["beta", "tau1", "tau2", "lambda"]
    if identity_term:
        dists.insert(2, Normal("y3", mean="beta", precision=ScaledMatrix(matrix="P3", scalar="tau3")))
        dists.append(Gamma("tau3", shape="a", rate="b"))
        state.update({"y3": y3, "P3": sparse.identity(p, format="csc"), "tau3": 1.0})
        names.insert(3, "tau3")
    mdl = Model(dists)
    samplers = [NormalNormal("beta", mdl)] + [NormalGamma(k, mdl) for k in names[1:]]
    with Streams(seed + 1) as s:
        M = _run_ref(state, samplers, mdl, n_iter)
    g = s.stack("g")[:, 0].reshape(n_iter, len(names) - 1)
    out = {"X1": X1, "X2": X2, "y1": y1, "y2": y2, "y3": y3, "w2": w2, "P_lambda": P_lambda.toarray(), "z": s.stack("z"),
           "identity_term": identity_term, "gmrf_prior": gmrf_prior, "names": np.array(names),
           "store_beta": M.store["beta"], "store_log_post": M.store["log_post"]}
    for j, k in enumerate(names[1:]):
        out["g_" + k] = g[:, j]
        out["store_" + k] = M.store[k]
    return out


def _run_ref(state, samplers, mdl, n_iter):
    import openmcmc.mcmc as m

    m.tqdm = lambda it: it
    M = MCMC(state, samplers, model=mdl, n_burn=0, n_iter=n_iter)
    M.run_mcmc()
    return M


def poisson_gamma_state(p, seed, layout="col", vector_prior=False):
    rng = np.random.default_rng(seed)
    lam_true = rng.gamma(5.0, 1.0, size=p)
    y = rng.poisson(lam_true).astype(float)
    shape = (p, 1) if layout == "col" else (1, p)
    a = np.full((p, 1), 2.0) + (rng.random((p, 1)) if vector_prior else 0.0)
    b = np.full((p, 1), 0.5) + (rng.random((p, 1)) * 0.2 if vector_prior else 0.0)
    if not vector_prior or layout != "col":
        a, b = np.array([[2.0]]), np.array([[0.5]])
    state = {"y": y.reshape(shape), "lam": (y + 1.0).reshape(shape) * 0.9, "a": a, "b": b}
    mdl = Model([Poisson("y", rate="lam"), Gamma("lam", shape="a", rate="b")])
    return state, mdl


def mmala_poisson_gamma_case(p, seed, n_iter, step, vector_prior=False):
    """mMALA on Poisson counts with a Gamma prior: the reference differentiates by finite differences (SURVEY F2/F3)."""
    state, mdl = poisson_gamma_state(p, seed, vector_prior=vector_prior)
    state0 = {k: np.array(v, copy=True) for k, v in state.items()}
    g0, H0 = mdl.grad_log_p(state0, "lam", hessian_required=True)
    lp0 = mdl.log_p(state0)
    with Streams(seed + 10) as s:
        smp = ManifoldMALA("lam", mdl, step=np.array([[step]]))
        M = _run_ref(state, [smp], mdl, n_iter)
    return {"y": state0["y"], "lam0": state0["lam"], "a": state0["a"], "b": state0["b"], "step": step,
            "grad0": g0, "hess0": H0, "logp0": lp0, "z": s.stack("z"), "u": s.stack("u").ravel(),
            "store_lam": M.store["lam"], "store_log_post": M.store["log_post"],
            "accept": np.array([smp.accept_rate.count["accept"], smp.accept_rate.count["proposal"]])}


def mmala_normal_case(p, seed, n_iter, step):
    """mMALA on a Normal prior + Normal 'observation' of theta: analytic derivatives in the reference, so the chain
    must replay to 1e-9."""
    rng = np.random.default_rng(seed)
    A = rng.standard_normal((p, p))
    P = A @ A.T + p * np.eye(p)
    state = {"theta": rng.standard_normal((p, 1)), "mu": rng.standard_normal((p, 1)), "P": P, "lam": 0.7,
             "yobs": rng.standard_normal((p, 1)), "W": sparse.diags(rng.random(p) + 0.5, format="csc"), "tau": 2.5}
    mdl = Model([Normal("theta", mean="mu", precision=ScaledMatrix(matrix="P", scalar="lam")),
                 Normal("yobs", mean="theta", precision=ScaledMatrix(matrix="W", scalar="tau"))])
    state0 = {k: (v.copy() if hasattr(v, "copy") else v) for k, v in state.items()}
    g0, H0 = mdl.grad_log_p({**state0, "lam": np.array([[0.7]]), "tau": np.array([[2.5]])}, "theta", hessian_required=True)
    with Streams(seed + 10) as s:
        smp = ManifoldMALA("theta", mdl, step=np.array([[step]]))
        M = _run_ref(state, [smp], mdl, n_iter)
    return {"theta0": state0["theta"], "mu": state0["mu"], "P": P, "lam": 0.7, "yobs": state0["yobs"],
            "w": np.asarray(state0["W"].diagonal()), "tau": 2.5, "step": step, "grad0": g0, "hess0": np.asarray(H0),
            "z": s.stack("z"), "u": s.stack("u").ravel(), "store_theta": M.store["theta"],
            "store_log_post": M.store["log_post"],
            "accept": np.array([smp.accept_rate.count["accept"], smp.accept_rate.count["proposal"]])}


def lognormal_case(p, seed, n_iter, step, sampler="mmala", prior="dense"):
    """SURVEY f4: theta ~ LogNormal(mu, (lam P)^-1) observed through yobs ~ N(theta, (tau W)^-1); every derivative is
    analytic in the reference (location_scale.py:340-343, 383-399), so chains replay to 1e-9."""
    rng = np.random.default_rng(seed)
    if prior == "dense":
        A = rng.standard_normal((p, p))
        P = A @ A.T / p + np.eye(p)
    else:
        P = sparse.diags(rng.random(p) + 0.5, format="csc")
    theta0 = np.exp(0.3 * rng.standard_normal((p, 1)))
    state = {"theta": theta0.copy(), "mu": 0.2 * rng.standard_normal((p, 1)), "P": P, "lam": 1.3,
             "yobs": theta0 + 0.3 * rng.standard_normal((p, 1)), "W": sparse.diags(rng.random(p) + 0.5, format="csc"),
             "tau": 4.0}
    mdl = Model([LogNormal("theta", mean="mu", precision=ScaledMatrix(matrix="P", scalar="lam")),
                 Normal("yobs", mean="theta", precision=ScaledMatrix(matrix="W", scalar="tau"))])
    state0 = {k: (v.copy() if hasattr(v, "copy") else v) for k, v in state.items()}
    sc = {**state0, "lam": np.array([[1.3]]), "tau": np.array([[4.0]])}
    prior_only = Model([mdl["theta"]])
    g0, H0 = prior_only.grad_log_p(sc, "theta", hessian_required=True)
    lp0 = prior_only.log_p(sc)
    with Streams(seed + 10) as s:
        if sampler == "mmala":
            smp = ManifoldMALA("theta", mdl, step=np.array([[step]]))
        else:
            smp = RandomWalk("theta", mdl, step=np.array([[step]]))
        M = _run_ref(state, [smp], mdl, n_iter)
    return {"theta0": state0["theta"], "mu": state0["mu"], "P": (P.toarray() if sparse.issparse(P) else P),
            "prior": prior, "lam": 1.3, "yobs": state0["yobs"], "w": np.asarray(state0["W"].diagonal()), "tau": 4.0,
            "step": step, "sampler": sampler, "grad0": g0, "hess0": np.asarray(H0), "logp0": lp0,
            "z": s.stack("z"), "u": s.stack("u").ravel(), "store_theta": M.store["theta"],
            "store_log_post": M.store["log_post"],
            "accept": np.array([smp.accept_rate.count["accept"], smp.accept_rate.count["proposal"]])}


def mmala_regression_case(n, p, seed, n_iter, step, transform=False, weighted=True, lognormal=False):
    """SURVEY a4 / f4 in an MH sampler: beta enters the mean of y ~ N(X f(beta), (tau W)^-1) linearly (f = exp with
    LinearCombinationWithTransform), Normal prior on beta: the mean-parameter branch of Normal.grad_log_p
    (location_scale.py:234-250) with parameter.py:199-228 / 283-297; analytic in the reference."""
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, p))
    if transform:
        X = np.abs(X)
    beta_true = 0.5 * rng.standard_normal((p, 1))
    f_true = np.exp(beta_true) if transform else beta_true
    y = X @ f_true + 0.5 * rng.standard_normal((n, 1))
    if lognormal:      # round 2: LogNormal response, mean-parameter branch of LogNormal.grad_log_p (location_scale.py:344-347)
        y = np.exp(0.3 * y)
    W = sparse.diags(rng.random(n) + 0.5, format="csc") if weighted else sparse.identity(n, format="csc")
    A = rng.standard_normal((p, p))
    P = A @ A.T / p + np.eye(p)
    mean = (LinearCombinationWithTransform(form={"beta": "X"}, transform={"beta": True}) if transform
            else LinearCombination(form={"beta": "X"}))
    mdl = Model([(LogNormal if lognormal else Normal)("y", mean=mean, precision=ScaledMatrix(matrix="W", scalar="tau")),
                 Normal("beta", mean="mu", precision=ScaledMatrix(matrix="P", scalar="lam"))])
    state = {"y": y, "X": X, "beta": beta_true + 0.1 * rng.standard_normal((p, 1)), "W": W, "tau": 1.7,
             "mu": np.zeros((p, 1)), "P": P, "lam": 0.8}
    state0 = {k: (v.copy() if hasattr(v, "copy") else v) for k, v in state.items()}
    sc = {**state0, "lam": np.array([[0.8]]), "tau": np.array([[1.7]])}
    lik_only = Model([mdl["y"]])
    g0, H0 = lik_only.grad_log_p(sc, "beta", hessian_required=True)
    lp0 = lik_only.log_p(sc)
    with Streams(seed + 10) as s:
        smp = ManifoldMALA("beta", mdl, step=np.array([[step]]))
        M = _run_ref(state, [smp], mdl, n_iter)
    return {"X": X, "y": y, "beta0": state0["beta"], "w": np.asarray(W.diagonal()), "weighted": weighted, "tau": 1.7,
            "P": P, "lam": 0.8, "transform": transform, "lognormal": lognormal, "step": step, "grad0": g0, "hess0": np.asarray(H0), "logp0": lp0,
            "z": s.stack("z"), "u": s.stack("u").ravel(), "store_beta": M.store["beta"],
            "store_log_post": M.store["log_post"],
            "accept": np.array([smp.accept_rate.count["accept"], smp.accept_rate.count["proposal"]])}


def rwl_case(p, seed, n_iter, step):
    """RandomWalkLoop over a (1, p) parameter with truncated proposals on [0, inf) (SURVEY F5: the only working form)."""
    state, mdl = poisson_gamma_state(p, seed, layout="row")
    state0 = {k: np.array(v, copy=True) for k, v in state.items()}
    with Streams(seed + 10) as s:
        smp = RandomWalkLoop("lam", mdl, step=np.array([[step]]), domain_limits=np.array([[0.0, np.inf]]),
                             max_variable_size=(1, p))   # a (1, p) parameter cannot be stored otherwise (sampler.py:107)
        M = _run_ref(state, [smp], mdl, n_iter)
    return {"y": state0["y"], "lam0": state0["lam"], "a": state0["a"], "b": state0["b"], "step": step,
            "limits": np.array([[0.0, np.inf]]), "tn_u": s.stack("tn_u").reshape(n_iter, p),
            "u": s.stack("u").reshape(n_iter, p), "store_lam": M.store["lam"], "store_log_post": M.store["log_post"],
            "accept": np.array([smp.accept_rate.count["accept"], smp.accept_rate.count["proposal"]])}


def rw_case(p, seed, n_iter, truncated):
    """RandomWalk (all elements at once): untruncated vector step, or truncated scalar."""
    state, mdl = poisson_gamma_state(p, seed, vector_prior=not truncated)
    state0 = {k: np.array(v, copy=True) for k, v in state.items()}
    rng = np.random.default_rng(seed + 5)
    step = np.array([[0.4]]) if truncated else 0.15 + 0.2 * rng.random((p, 1))
    lim = np.array([[0.5, 12.0]]) if truncated else None
    with Streams(seed + 10) as s:
        smp = RandomWalk("lam", mdl, step=step, domain_limits=lim)
        M = _run_ref(state, [smp], mdl, n_iter)
    return {"y": state0["y"], "lam0": state0["lam"], "a": state0["a"], "b": state0["b"], "step": step,
            "limits": lim if truncated else np.zeros((0, 2)),
            "z": (s.stack("tn_u") if truncated else s.stack("z")).reshape(n_iter, p), "u": s.stack("u").ravel(),
            "store_lam": M.store["lam"], "store_log_post": M.store["log_post"],
            "accept": np.array([smp.accept_rate.count["accept"], smp.accept_rate.count["proposal"]])}


def truncnorm_grid(seed=0, n=400):
    """scipy.stats.truncnorm ppf / logpdf on random and tail cases (what gmrf.py:269-318 calls)."""
    rng = np.random.default_rng(seed)
    mean = rng.normal(size=n) * 3
    scale = rng.random(n) * 2 + 0.05
    lower = mean + scale * rng.normal(size=n) * 3
    upper = lower + rng.random(n) * 5 * scale + 1e-3
    upper[rng.random(n) < 0.3] = np.inf
    lower[rng.random(n) < 0.2] = -np.inf
    # far tails on both sides
    k = n // 8
    lower[:k] = mean[:k] + scale[:k] * (4 + 10 * rng.random(k))
    upper[:k] = np.inf
    upper[k:2 * k] = mean[k:2 * k] - scale[k:2 * k] * (4 + 10 * rng.random(k))
    lower[k:2 * k] = -np.inf
    u = rng.random(n)
    a, b = (lower - mean) / scale, (upper - mean) / scale
    x = stats.truncnorm.ppf(u, a, b, loc=mean, scale=scale)
    lp = gmrf.truncated_normal_log_pdf(x, mean, scale, lower, upper)
    x_other = np.clip(x + scale * rng.normal(size=n), np.where(np.isfinite(lower), lower, x - 1), np.where(np.isfinite(upper), upper, x + 1))
    lp_other = gmrf.truncated_normal_log_pdf(x_other, mean, scale, lower, upper)
    return {"mean": mean, "scale": scale, "lower": lower, "upper": upper, "u": u, "x": x, "logpdf": lp,
            "x_other": x_other, "logpdf_other": lp_other}


def mh_cases():
    return {
        "mmala_poisson_gamma_p6": mmala_poisson_gamma_case(6, 11, 8, 0.5),
        "mmala_poisson_gamma_p32_vec": mmala_poisson_gamma_case(32, 12, 3, 0.4, vector_prior=True),
        "mmala_normal_p7": mmala_normal_case(7, 13, 8, 0.8),
        "mmala_normal_p40": mmala_normal_case(40, 14, 4, 0.9),
        "rwl_poisson_gamma_1x8": rwl_case(8, 15, 6, 0.5),
        "rw_poisson_gamma_p6": rw_case(6, 16, 10, truncated=False),
        "rw_trunc_scalar": rw_case(1, 17, 12, truncated=True),
        "truncnorm_grid": truncnorm_grid(),
    }


def mh_f4_cases():
    return {
        "lognormal_mmala_p5_dense": lognormal_case(5, 21, 10, 0.7),
        "lognormal_mmala_p24_diag": lognormal_case(24, 22, 6, 0.3, prior="diag"),
        "lognormal_rw_p6_dense": lognormal_case(6, 23, 12, 0.08, sampler="rw"),
        "mhreg_mmala_n60_p6": mmala_regression_case(60, 6, 24, 10, 0.8),
        "mhreg_mmala_n200_p30_eye": mmala_regression_case(200, 30, 25, 4, 0.9, weighted=False),
        "mhreg_exp_mmala_n80_p5": mmala_regression_case(80, 5, 26, 10, 0.7, transform=True),
    }


# ----------------------------------------------------------------------------------------------- mixture model (SURVEY f2)
def mixture_case(n, p, n_cat, seed, n_iter, sample_mean=True, prob_rows=1):
    """The reference's standard mixture model (tests/test_sampler.py:113-147): y ~ N(X beta, W^-1), beta_i ~
    N(mu[z_i], 1/tau[z_i]), z_i ~ Cat(prob), tau_k ~ Gamma; optionally mu ~ N(m0, (lam0 I)^-1).  Samplers:
    NormalNormal(beta), [NormalNormal(mu)], NormalGamma(tau) with its K-loop, MixtureAllocation(z)."""
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, p))
    z_true = rng.integers(0, n_cat, size=(p, 1))
    mu_true = np.linspace(-3, 3, n_cat).reshape(n_cat, 1)
    beta_true = mu_true[z_true.ravel()] + 0.3 * rng.standard_normal((p, 1))
    y = X @ beta_true + 0.5 * rng.standard_normal((n, 1))
    W = sparse.diags(rng.random(n) + 0.5, format="csc")
    prob = rng.random((prob_rows, n_cat)) + 0.2
    prob = prob / prob.sum(axis=1, keepdims=True)
    dists = [Normal("y", mean=LinearCombination(form={"beta": "X"}), precision=Identity("W")),
             Normal("beta", mean=MixtureParameterVector(param="mu", allocation="z"),
                    precision=MixtureParameterMatrix(param="tau", allocation="z")),
             Gamma("tau", shape="a_tau", rate="b_tau"),
             Categorical("z", prob="prob")]
    if sample_mean:
        dists.append(Normal("mu", mean="m0", precision=ScaledMatrix(matrix="P_mu", scalar="lam0")))
    mdl = Model(dists)
    samplers = [NormalNormal("beta", mdl)]
    if sample_mean:
        samplers.append(NormalNormal("mu", mdl))
    samplers += [NormalGamma("tau", mdl), MixtureAllocation("z", mdl, response_param="beta")]
    state = {"y": y, "X": X, "W": W, "beta": np.zeros((p, 1)), "mu": mu_true + 0.5 * rng.standard_normal((n_cat, 1)),
             "tau": 1.0 + rng.random((n_cat, 1)), "z": rng.integers(0, n_cat, size=(p, 1)), "prob": prob,
             "a_tau": 2.0 * np.ones((n_cat, 1)), "b_tau": 0.5 + rng.random((n_cat, 1)),
             "m0": np.zeros((n_cat, 1)), "P_mu": sparse.identity(n_cat, format="csc"), "lam0": 0.1}
    state0 = {k: (v.copy() if hasattr(v, "copy") else v) for k, v in state.items()}
    with Streams(seed + 1) as s:
        M = _run_ref(state, samplers, mdl, n_iter)
    z_all = s.stack("z")                               # NormalNormal(beta) [p], then NormalNormal(mu) [n_cat] per sweep
    zb = np.array([r for r in s.log["z"] if r.size == p]) if p != n_cat else None
    zm = np.array([r for r in s.log["z"] if r.size == n_cat]) if sample_mean else np.zeros((0, n_cat))
    out = {"X": X, "y": y, "w": np.asarray(W.diagonal()), "prob": prob, "sample_mean": sample_mean,
           "beta0": state0["beta"], "mu0": state0["mu"], "tau0": state0["tau"], "z0": state0["z"].astype(float),
           "a_tau": state0["a_tau"], "b_tau": state0["b_tau"], "lam0": 0.1,
           "z_beta": zb, "z_mu": zm, "g": s.stack("g").reshape(n_iter, n_cat), "u": s.stack("u").reshape(n_iter, p),
           "store_beta": M.store["beta"], "store_tau": M.store["tau"], "store_z": M.store["z"].astype(float),
           "store_log_post": M.store["log_post"]}
    if sample_mean:
        out["store_mu"] = M.store["mu"]
    del z_all
    return out


def mixture_cases():
    return {
        "mixture_n80_p12_k3": mixture_case(80, 12, 3, 31, 6, sample_mean=False),
        "mixture_n60_p20_k4_rowprob": mixture_case(60, 20, 4, 32, 5, sample_mean=False, prob_rows=20),
    }


# ----------------------------------------------------------------------------------------------- temporal GMRF (C3 shape)
def gmrf_case(n, seed, n_iter, form="notebook", irregular=False, weighted=False, nonzero_mu=False,
              order=("b", "lambda", "tau")):
    """examples/4_GMRF_smoother: b ~ N(mu, (lambda P)^-1), y ~ N(b, (tau W)^-1), Gamma priors on lambda and tau.
    form="notebook": mean="b" (the reference then runs DENSE linear algebra, SURVEY F4);
    form="sparse"  : mean=LinearCombination({"b": "I"}) with sparse I (SuperLU path, gmrf.py:489-520)."""
    rng = np.random.default_rng(seed)
    s = np.arange(n) * (60.0 / 99.0)
    if irregular:
        s = np.cumsum(0.2 + rng.random(n))
    P = gmrf.precision_irregular(s)
    P[0, 0] = P[0, 0] + 0.001
    P = sparse.csc_matrix(P)
    truth = np.sin(s / 20) + 2 * np.cos(s / 12) + 2
    y = truth + rng.standard_normal(n)
    W = sparse.diags(rng.random(n) + 0.5, format="csc") if weighted else sparse.csc_matrix(np.eye(n))
    mu = (0.5 * rng.standard_normal(n) + 2.0) if nonzero_mu else np.zeros(n)
    mean = "b" if form == "notebook" else LinearCombination(form={"b": "I"})
    mdl = Model([Normal("y", mean=mean, precision=ScaledMatrix(matrix="P_tau", scalar="tau")),
                 Normal("b", mean="mu", precision=ScaledMatrix(matrix="P_lambda", scalar="lambda")),
                 Gamma("lambda", shape="a_lam", rate="b_lam"),
                 Gamma("tau", shape="a_tau", rate="b_tau")])
    state = {"y": y.copy(), "b": y.copy(), "mu": mu, "lambda": 100, "P_lambda": P, "a_lam": 10, "b_lam": 1, "tau": 1,
             "P_tau": W, "a_tau": 1, "b_tau": 1}
    if form != "notebook":
        state["I"] = sparse.identity(n, format="csc")
    smap = {"b": NormalNormal("b", mdl), "lambda": NormalGamma("lambda", mdl), "tau": NormalGamma("tau", mdl)}
    with Streams(seed + 1) as st:
        M = _run_ref(state, [smap[k] for k in order], mdl, n_iter)
    g = st.stack("g")
    gorder = [k for k in order if k != "b"]
    Pc = P.tocsc()
    return {"s": s, "y": y, "mu": mu, "pd": Pc.diagonal(), "pe": Pc.diagonal(1), "w": np.asarray(W.diagonal()),
            "form": form, "order": np.array(order), "z": st.stack("z"),
            "g_" + gorder[0]: g[0::2, 0], "g_" + gorder[1]: g[1::2, 0],
            "store_b": M.store["b"], "store_lambda": M.store["lambda"], "store_tau": M.store["tau"],
            "store_log_post": M.store["log_post"]}


def gmrf_cases():
    return {
        "gmrf_n100_notebook": gmrf_case(100, 21, 5),
        "gmrf_n100_sparse": gmrf_case(100, 21, 5, form="sparse"),
        "gmrf_n2500_sparse_weighted_mu": gmrf_case(2500, 22, 3, form="sparse", weighted=True, nonzero_mu=True,
                                                   order=("tau", "b", "lambda")),
        "gmrf_n5000_sparse_irregular": gmrf_case(5000, 23, 3, form="sparse", irregular=True),
    }


# ----------------------------------------------------------------------------------------------- reversible jump (C5)
def _rj_basis(X, theta, omega):
    """tests/test_reversible_jump.py:23-40 of the reference (make_basis), restated for the state update callbacks."""
    B = np.full((X.shape[0], theta.shape[1]), np.nan)
    for k in range(theta.shape[1]):
        B[:, [k]] = stats.norm.pdf(X, loc=theta[:, k], scale=omega[:, k])
    return B


def rj_case(seed, n_data, n0, n_max, n_steps, response="normal", with_omega=True, limits=(-10.0, 10.0), rho=6.0,
            birth_probability=0.5):
    """The reference's own RJ test model (tests/test_reversible_jump.py:137-252) driven step by step: only the
    ReversibleJump sampler runs; every step records the state before, the variates, the proposal and the outcome."""
    import openmcmc.sampler.reversible_jump as rjmod

    rng = np.random.default_rng(seed)
    lo, hi = -10.0, 10.0
    X = lo + (hi - lo) * np.sort(rng.random((n_data, 1)), axis=0)
    theta = lo + (hi - lo) * rng.random((1, n0))
    omega = 0.7 + 0.8 * rng.random((1, n0)) if with_omega else np.ones((1, n0))
    B = _rj_basis(X, theta, omega)
    tau_beta, tau_y = 0.25, 100.0
    beta = 2.0 * rng.standard_normal((n0, 1))
    y = B @ beta + 0.1 * rng.standard_normal((n_data, 1))
    state = {"y": y, "beta": beta + 0.05 * rng.standard_normal((n0, 1)), "tau_y": np.array([[tau_y]]), "P": sparse.eye(n_data), "B": B,
             "n_basis": np.array([[float(n0)]]), "X": X, "theta": theta, "omega": omega, "mu_beta": np.zeros((1, 1)),
             "tau_beta": tau_beta * np.ones((1, 1)), "rho": np.array([[rho]]), "alloc_beta": np.zeros((n0, 1), dtype=int),
             "a_omega": 3.0 * np.ones((1, 1)), "b_omega": 2.0 * np.ones((1, 1))}
    mean = LinearCombination(form={"beta": "B"})
    prec = ScaledMatrix(matrix="P", scalar="tau_y")
    resp = (Normal if response == "normal" else NullDistribution)(response="y", mean=mean, precision=prec)
    dists = [resp,
             Normal(response="beta", mean=MixtureParameterVector(param="mu_beta", allocation="alloc_beta"),
                    precision=MixtureParameterMatrix(param="tau_beta", allocation="alloc_beta")),
             Poisson(response="n_basis", rate="rho"),
             Uniform(response="theta", domain_response_lower=np.array([lo], ndmin=2),
                     domain_response_upper=np.array([hi], ndmin=2))]
    assoc = ["theta"]
    if with_omega:
        dists.append(Gamma("omega", shape="a_omega", rate="b_omega"))
        assoc.append("omega")
    mdl = Model(dists)

    def birth_fn(current_state, prop_state):
        if not with_omega:
            prop_state["omega"] = np.concatenate((prop_state["omega"], prop_state["omega"][:, -1:]), axis=1)
        prop_state["B"] = _rj_basis(prop_state["X"], prop_state["theta"], prop_state["omega"])
        prop_state["alloc_beta"] = np.concatenate((prop_state["alloc_beta"], np.array([0], ndmin=2)), axis=0)
        return prop_state, 0.0, 0.0

    def death_fn(current_state, prop_state, deletion_index):
        if not with_omega:
            prop_state["omega"] = np.delete(prop_state["omega"], obj=deletion_index, axis=1)
        prop_state["B"] = np.delete(prop_state["B"], obj=deletion_index, axis=1)
        prop_state["alloc_beta"] = np.delete(prop_state["alloc_beta"], obj=deletion_index, axis=0)
        return prop_state, 0.0, 0.0

    matching = {"variable": "beta", "matrix": "B", "scale": 1.0, "limits": list(limits) if limits else None}
    rj = ReversibleJump(param="n_basis", model=mdl, associated_params=assoc, n_max=n_max, state_birth_function=birth_fn,
                        state_death_function=death_fn, matching_params=matching, birth_probability=birth_probability)
    keys = ["n", "theta", "omega", "beta"]
    rec = {k + "_before": [] for k in keys}
    rec.update({k + "_after": [] for k in keys})
    for k in ("birth", "del_index", "u_move", "theta_new", "omega_new", "beta_new", "u_accept", "lq_fwd", "lq_rev",
              "log_accept", "accepted", "cond"):
        rec[k] = []

    def pad(a):
        out = np.full(n_max, np.nan)
        a = np.asarray(a, dtype=float).ravel()
        out[: a.size] = a
        return out

    info = {}
    orig_prop = rj.proposal
    orig_acc = rj.accept_proposal

    def prop(current_state, param_index=None):
        out = orig_prop(current_state)
        info.update(prop=out[0], lq_fwd=out[1], lq_rev=out[2])
        return out

    def acc(log_accept):
        r = orig_acc(log_accept)
        info.update(log_accept=log_accept, accepted=r)
        return r

    rj.proposal = prop
    rj.accept_proposal = acc
    with Streams(seed + 1000) as S:
        for it in range(n_steps):
            n = int(np.asarray(state["n_basis"]).ravel()[0])
            for k, v in (("n", [n]), ("theta", state["theta"]), ("omega", state["omega"]), ("beta", state["beta"])):
                rec[k + "_before"].append(pad(v) if k != "n" else float(n))
            nu, nr = len(S.log["u"]), len(S.log["randint"])
            sB = state["B"]
            state = rj.sample(state)
            us = [float(u.ravel()[0]) for u in S.log["u"][nu:]]
            birth = int(np.asarray(info["prop"]["n_basis"]).ravel()[0]) == n + 1
            edge = n in (1, n_max)
            rec["birth"].append(float(birth))
            rec["u_move"].append(np.nan if edge else us[0])
            rec["u_accept"].append(us[-1])
            rec["del_index"].append(-1.0 if birth else float(S.log["randint"][nr][0]))
            rec["theta_new"].append(float(info["prop"]["theta"][0, -1]) if birth else np.nan)
            rec["omega_new"].append(float(info["prop"]["omega"][0, -1]) if birth else np.nan)
            rec["beta_new"].append(float(info["prop"]["beta"][-1, 0]) if birth else np.nan)
            for k in ("lq_fwd", "lq_rev", "log_accept"):
                rec[k].append(float(np.asarray(info[k]).ravel()[0]))
            rec["accepted"].append(float(info["accepted"]))
            Bc = info["prop"]["B"] if birth else sB
            rec["cond"].append(float(np.linalg.cond(Bc.T @ Bc + 1e-10 * np.eye(Bc.shape[1]))))
            for k, v in (("n", None), ("theta", state["theta"]), ("omega", state["omega"]), ("beta", state["beta"])):
                rec[k + "_after"].append(pad(v) if k != "n" else float(np.asarray(state["n_basis"]).ravel()[0]))
    out = {k: np.array(v) for k, v in rec.items()}
    out.update(X=X.ravel(), y=y.ravel(), tau_y=tau_y, tau_beta=tau_beta, mu_beta=0.0, rho=rho, a_omega=3.0, b_omega=2.0,
               theta_lo=lo, theta_hi=hi, n_max=n_max, birth_probability=birth_probability, match_scale=1.0,
               match_limits=np.array(limits if limits else [np.nan, np.nan]), response=response,
               with_omega=float(with_omega))
    return out


def rj_companion_case(seed, n_data, n0, n_max, n_sweeps, response="normal"):
    """The other three samplers of the reference's RJ model (tests/test_reversible_jump.py:213-252) driven call by call
    on states whose size the (unrecorded) ReversibleJump steps in between keep changing: ManifoldMALA on beta,
    RandomWalkLoop on theta and on omega with move_function = make_basis as state_update_function.  Every call records
    the state before, its variates and the state after."""
    rng = np.random.default_rng(seed)
    lo, hi, wlo, whi = -10.0, 10.0, 0.5, 2.0
    X = lo + (hi - lo) * np.sort(rng.random((n_data, 1)), axis=0)
    theta = lo + (hi - lo) * rng.random((1, n0))
    omega = 0.7 + 0.8 * rng.random((1, n0))
    B = _rj_basis(X, theta, omega)
    tau_beta, tau_y, rho = 0.25, 100.0, float(n0)
    beta = 2.0 * rng.standard_normal((n0, 1))
    y = B @ beta + 0.1 * rng.standard_normal((n_data, 1))
    state = {"y": y, "beta": beta + 0.05 * rng.standard_normal((n0, 1)), "tau_y": np.array([[tau_y]]), "P": sparse.eye(n_data),
             "B": B, "n_basis": np.array([[float(n0)]]), "X": X, "theta": theta, "omega": omega, "mu_beta": np.zeros((1, 1)),
             "tau_beta": tau_beta * np.ones((1, 1)), "rho": np.array([[rho]]), "alloc_beta": np.zeros((n0, 1), dtype=int),
             "a_omega": 3.0 * np.ones((1, 1)), "b_omega": 2.0 * np.ones((1, 1))}
    mean = LinearCombination(form={"beta": "B"})
    prec = ScaledMatrix(matrix="P", scalar="tau_y")
    resp = (Normal if response == "normal" else NullDistribution)(response="y", mean=mean, precision=prec)
    mdl = Model([resp,
                 Normal(response="beta", mean=MixtureParameterVector(param="mu_beta", allocation="alloc_beta"),
                        precision=MixtureParameterMatrix(param="tau_beta", allocation="alloc_beta")),
                 Poisson(response="n_basis", rate="rho"),
                 Uniform(response="theta", domain_response_lower=np.array([lo], ndmin=2),
                         domain_response_upper=np.array([hi], ndmin=2)),
                 Gamma("omega", shape="a_omega", rate="b_omega")])

    def move_fn(st, param_index):
        st["B"] = _rj_basis(st["X"], st["theta"], st["omega"])
        return st, 0.0, 0.0

    def birth_fn(current_state, prop_state):
        prop_state["B"] = _rj_basis(prop_state["X"], prop_state["theta"], prop_state["omega"])
        prop_state["alloc_beta"] = np.concatenate((prop_state["alloc_beta"], np.array([0], ndmin=2)), axis=0)
        return prop_state, 0.0, 0.0

    def death_fn(current_state, prop_state, deletion_index):
        prop_state["B"] = np.delete(prop_state["B"], obj=deletion_index, axis=1)
        prop_state["alloc_beta"] = np.delete(prop_state["alloc_beta"], obj=deletion_index, axis=0)
        return prop_state, 0.0, 0.0

    step_b, step_t, step_w = 0.5, 0.3, 0.1
    mmala = ManifoldMALA(param="beta", model=mdl, step=np.array(step_b), max_variable_size=n_max)
    rw_t = RandomWalkLoop(param="theta", model=mdl, step=np.array(step_t), max_variable_size=n_max,
                          domain_limits=np.array([lo, hi], ndmin=2), state_update_function=move_fn)
    rw_w = RandomWalkLoop(param="omega", model=mdl, step=np.array(step_w), max_variable_size=n_max,
                          domain_limits=np.array([wlo, whi], ndmin=2), state_update_function=move_fn)
    rj = ReversibleJump(param="n_basis", model=mdl, associated_params=["theta", "omega"], n_max=n_max,
                        state_birth_function=birth_fn, state_death_function=death_fn,
                        matching_params={"variable": "beta", "matrix": "B", "scale": 1.0, "limits": [-10.0, 10.0]})

    def pad(a):
        out = np.zeros(n_max)
        a = np.asarray(a, dtype=float).ravel()
        out[: a.size] = a
        return out

    rec = {k: [] for k in ("kind", "n", "theta_before", "omega_before", "beta_before", "theta_after", "omega_after",
                           "beta_after", "z", "tn_u", "u", "accepted")}
    kinds = {"beta": 0, "theta": 1, "omega": 2}
    for it in range(n_sweeps):
        for smp in (mmala, rw_t, rw_w):
            n = int(np.asarray(state["n_basis"]).ravel()[0])
            before = {k: pad(state[k]) for k in ("theta", "omega", "beta")}
            a0 = smp.accept_rate.count["accept"]
            with Streams(seed + 77 * it + kinds[smp.param]) as S:
                state = smp.sample(state)
            rec["kind"].append(float(kinds[smp.param]))
            rec["n"].append(float(n))
            for k in ("theta", "omega", "beta"):
                rec[k + "_before"].append(before[k])
                rec[k + "_after"].append(pad(state[k]))
            rec["z"].append(pad(np.concatenate(S.log["z"])) if S.log["z"] else np.zeros(n_max))
            rec["tn_u"].append(pad(np.concatenate(S.log["tn_u"])) if S.log["tn_u"] else np.zeros(n_max))
            rec["u"].append(pad(np.concatenate(S.log["u"])))
            rec["accepted"].append(float(smp.accept_rate.count["accept"] - a0))
        with Streams(seed + 5000 + it):
            state = rj.sample(state)      # unrecorded: changes the size of the state between the recorded calls
    out = {k: np.array(v) for k, v in rec.items()}
    out.update(X=X.ravel(), y=y.ravel(), tau_y=tau_y, tau_beta=tau_beta, mu_beta=0.0, rho=rho, a_omega=3.0, b_omega=2.0,
               theta_lo=lo, theta_hi=hi, omega_lo=wlo, omega_hi=whi, n_max=n_max, step_beta=step_b, step_theta=step_t,
               step_omega=step_w, response=response)
    return out


def rj_cases():
    return {
        "rj_normal_n50_k4": rj_case(0, 50, 4, 12, 60),
        "rj_null_n50_k4": rj_case(1, 50, 4, 8, 80, response="null", rho=4.0),
        "rj_normal_untruncated_fixed_width": rj_case(2, 40, 3, 10, 50, with_omega=False, limits=None),
        "rj_edges_nmax3": rj_case(3, 30, 1, 3, 60, response="null", rho=2.0, birth_probability=0.4),
    }


def replicated_case(dim, n_rep, seed, n_iter, scaled=False):
    """The model of the reference's examples 1 and 2 (y of shape (dim, n_rep): replicates in columns, Identity mean):
    log_p / gradient / Hessian at the start state, a RandomWalk chain and a NormalNormal chain on the mean."""
    rng = np.random.default_rng(seed)
    h_true = 160 + 10 * rng.standard_normal((dim, 1))
    y = h_true + 12 * rng.standard_normal((dim, n_rep))
    pdiag = 0.5 + rng.random(dim)
    if scaled:
        prec = ScaledMatrix(matrix="P", scalar="tau")
        extra = {"P": sparse.diags([pdiag], [0], format="csc"), "tau": np.array(1 / 150, ndmin=2)}
    else:
        prec = "tau"
        extra = {"tau": np.array(1 / 200, ndmin=2) if dim == 1 else np.diag(pdiag / 150)}
    mdl = Model([Normal("y", mean="h", precision=prec), Normal("h", mean="mu", precision="lambda")])
    state = {"y": y, "h": 200.0 * np.ones((dim, 1)), "mu": 160.0 * np.ones((dim, 1)),
             "lambda": np.array(1 / 100, ndmin=2) if dim == 1 else np.eye(dim) / 100, **extra}
    state0 = {k: (v.copy() if hasattr(v, "copy") else v) for k, v in state.items()}
    out = {"y": y, "h0": state0["h"], "mu": state0["mu"], "lam": np.asarray(state0["lambda"]), "pdiag": pdiag,
           "tau": np.asarray(state0["tau"]), "scaled": np.array(int(scaled)), "logp0": np.array(mdl.log_p(state))}
    g, H = mdl.grad_log_p(state, "h")
    out["grad0"], out["hess0"] = np.asarray(g), np.asarray(H.todense() if sparse.issparse(H) else H)
    with Streams(seed + 1) as s:
        smp = RandomWalk("h", mdl, step=np.array([[4.0]]))
        M = _run_ref({k: (v.copy() if hasattr(v, "copy") else v) for k, v in state0.items()}, [smp], mdl, n_iter)
    out.update({"rw_z": s.stack("z").reshape(n_iter, dim), "rw_u": s.stack("u").ravel(), "rw_store_h": M.store["h"],
                "rw_store_log_post": M.store["log_post"],
                "rw_accept": np.array([smp.accept_rate.count["accept"], smp.accept_rate.count["proposal"]])})
    with Streams(seed + 2) as s:
        M = _run_ref({k: (v.copy() if hasattr(v, "copy") else v) for k, v in state0.items()}, [NormalNormal("h", mdl)],
                     mdl, n_iter)
    out.update({"nn_z": s.stack("z").reshape(n_iter, dim), "nn_store_h": M.store["h"],
                "nn_store_log_post": M.store["log_post"]})
    return out


def replicated_regression_case(dim, p, n_rep, seed, n_iter):
    """Round 2: replicates in the columns of y with a LinearCombination mean -- y[:, r] ~ N(X beta, (tau W)^-1) for every
    column r (distribution.py:8-10; the n_rep factor of location_scale.py:238-241): log_p / gradient / Hessian at the
    start state and a ManifoldMALA chain on beta (the reference's conjugate samplers do not take this form:
    sampler.py:192 fails to broadcast)."""
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((dim, p))
    beta_true = rng.standard_normal((p, 1))
    y = X @ beta_true + 0.4 * rng.standard_normal((dim, n_rep))
    W = sparse.diags(rng.random(dim) + 0.5, format="csc")
    mdl = Model([Normal("y", mean=LinearCombination(form={"beta": "X"}), precision=ScaledMatrix(matrix="W", scalar="tau")),
                 Normal("beta", mean="mu", precision=ScaledMatrix(matrix="P", scalar="lam")),
                 Gamma("tau", shape="a", rate="b")])
    state = {"y": y, "X": X, "beta": np.zeros((p, 1)), "W": W, "tau": 1.5, "mu": np.zeros((p, 1)),
             "P": sparse.identity(p, format="csc"), "lam": 0.3, "a": 2.0, "b": 1.0}
    state0 = {k: (v.copy() if hasattr(v, "copy") else v) for k, v in state.items()}
    sc = {**state0, "tau": np.array([[1.5]]), "lam": np.array([[0.3]]), "a": np.array([[2.0]]), "b": np.array([[1.0]])}
    lik = Model([mdl["y"]])
    g0, H0 = lik.grad_log_p(sc, "beta", hessian_required=True)
    out = {"X": X, "y": y, "w": np.asarray(W.diagonal()), "tau": 1.5, "lam": 0.3, "a": 2.0, "b": 1.0,
           "logp0": np.array(lik.log_p(sc)), "grad0": np.asarray(g0), "hess0": np.asarray(H0.todense() if sparse.issparse(H0) else H0)}
    with Streams(seed + 1) as s:
        smp = ManifoldMALA("beta", mdl, step=np.array([[0.8]]))
        M = _run_ref(state, [smp], mdl, n_iter)
    out.update({"z": s.stack("z"), "u": s.stack("u").ravel(), "store_beta": M.store["beta"],
                "store_log_post": M.store["log_post"], "beta0": state0["beta"],
                "accept": np.array([smp.accept_rate.count["accept"], smp.accept_rate.count["proposal"]])})
    return out


def main():
    cases = {
        "regression_n50_p3": regression_case(50, 3, 0, 6),
        "regression_n200_p8_weighted_diag": regression_case(200, 8, 1, 4, weighted=True, prior="diag"),
        "regression_n300_p17_dense_reordered": regression_case(300, 17, 2, 4, order=("tau", "lambda", "beta"),
                                                               prior="dense"),
        "regression_n1000_p64": regression_case(1000, 64, 3, 3),
        "truncreg_n120_p6_two_sided": regression_case(120, 6, 4, 5, trunc=(np.array([[-0.2]]), np.array([[0.6]]))),
        "truncreg_n80_p40_upper_dense": regression_case(80, 40, 5, 3, prior="dense", weighted=True,
                                                        trunc=(None, np.array([[0.25]]))),
        "truncreg_n30_p1_lower": regression_case(30, 1, 6, 6, trunc=(np.array([[0.5]]), None)),
        "twoterm_n150_p7_q4": regression_two_term_case(150, 7, 4, 7, 5),
    }
    which = sys.argv[1:] or ["regression", "mh", "mh_f4", "mixture", "gmrf", "rj", "rj_moves", "replicated", "round2", "round2b", "round2c", "round2d"]
    if "regression" not in which:
        cases = {}
    if "round2" in which:
        # round 2: high signal-to-noise (the re-centred rss must not cancel), p > 64 (blocked Cholesky, column panels),
        # RandomWalkLoop at the BASELINE C4b width (1, 32)
        cases.update({
            "regression_n400_p12_highsnr": regression_case(400, 12, 21, 5, noise=1e-4),
            "regression_n600_p128": regression_case(600, 128, 22, 3),
            "regression_n700_p200_dense_weighted": regression_case(700, 200, 23, 2, weighted=True, prior="dense"),
            "rwl_poisson_gamma_1x32": rwl_case(32, 24, 6, 0.5),
        })
    if "round2b" in which:
        # round 2: NormalNormal with several likelihood terms / an Identity-mean term / a tridiagonal prior on regression
        # coefficients (sampler.py:179-192)
        cases.update({
            "multilik_n90_n60_p7_identity": multilik_case(90, 60, 7, 31, 5),
            "multilik_n200_n150_p40": multilik_case(200, 150, 40, 32, 3, identity_term=False),
            "multilik_gmrfprior_n120_n80_p24": multilik_case(120, 80, 24, 33, 4, identity_term=True, gmrf_prior=True),
        })
    if "round2c" in which:
        # round 2: LogNormal response with a LinearCombination mean inside ManifoldMALA (mean-parameter branch)
        cases.update({"mhreg_lognormal_mmala_n70_p5": mmala_regression_case(70, 5, 27, 10, 0.8, lognormal=True),
                      "mhreg_lognormal_mmala_n150_p20_eye": mmala_regression_case(150, 20, 28, 5, 0.9, weighted=False,
                                                                                  lognormal=True)})
    if "round2d" in which:
        cases.update({"replicated_regression_d40_p5_r6": replicated_regression_case(40, 5, 6, 61, 6),
                      "replicated_regression_d9_p3_r25": replicated_regression_case(9, 3, 25, 62, 8)})
    if "mh" in which:
        cases.update(mh_cases())
    if "mh_f4" in which:
        cases.update(mh_f4_cases())
    if "mixture" in which:
        cases.update(mixture_cases())
    if "gmrf" in which:
        cases.update(gmrf_cases())
    if "rj" in which:
        cases.update(rj_cases())
    if "rj_moves" in which:
        cases.update({"rjmoves_normal_n60_k5": rj_companion_case(41, 60, 5, 12, 6),
                      "rjmoves_null_n40_k3": rj_companion_case(42, 40, 3, 8, 5, response="null")})
    if "replicated" in which:
        cases.update({"replicated_d1_r5": replicated_case(1, 5, 51, 8),
                      "replicated_d3_r7_scaled": replicated_case(3, 7, 52, 6, scaled=True),
                      "replicated_d2_r4_diag": replicated_case(2, 4, 53, 6)})
    for name, d in cases.items():
        np.savez_compressed(os.path.join(OUT, name + ".npz"), **d)
        print("wrote", name, {k: np.shape(v) for k, v in d.items() if k.startswith("store")})


if __name__ == "__main__":
    main()
