"""GPU: ManifoldMALA above 64 parameters -- the blocked dense step (64 < p <= 512, mmala_blocked_kernel) and the
element-wise step (64 < n <= 4096, mmala_diag_wide_kernel) -- against the numpy oracle (oracle/mh.py: mmala_step, the
function the mmala_* / mhreg_* goldens of the live reference pin at p <= 40) with injected z / u, through MCMC, free
running against closed-form posteriors, and at their edges (chain slices, failures, refusals).

Bars: probes mu / L rel 1e-10, proposal / scalars / states rel 1e-9, accept decisions exact.  The oracle factors the
dense Hessian in numpy, so its cost sets the number of chains checked at the largest sizes."""

import numpy as np
import pytest
from scipy import sparse, stats

pytestmark = pytest.mark.gpu


def _dev(x):
    import torch

    return torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64)).cuda()


def _spd(rng, p, scale=1.0):
    B = rng.standard_normal((p, p))
    return np.eye(p) + scale * (B @ B.T) / p


# ------------------------------------------------------------------------------------------------ model builders
def _dense_case(kind, p, C, seed):
    """Per-chain data for one dense-Hessian model: (device terms, keep-alive tensors, theta0 (C, p), oracle terms per
    chain, step)."""
    from openmcmc_b200 import kernels as K
    from oracle import mh

    rng = np.random.default_rng(seed)
    keep, oterms = [], [[] for _ in range(C)]

    def dv(x):
        t = _dev(x)
        keep.append(t)
        return t

    P = np.stack([_spd(rng, p) for _ in range(C)])
    logdetP = np.array([np.linalg.slogdet(P[c])[1] for c in range(C)])
    terms = []
    if kind in ("linear", "linear_exp"):
        tr = kind == "linear_exp"
        nd, lam, tau = p + 16, 1.0, 4.0
        X = rng.standard_normal((C, nd, p)) / np.sqrt(p)
        bt = 0.1 * rng.standard_normal((C, p, 1))
        y = X @ (np.exp(bt) if tr else bt) + 0.2 * rng.standard_normal((C, nd, 1))
        rec = np.concatenate([np.einsum("cni,cnj->cij", X, X).reshape(C, -1), np.einsum("cni,cn->ci", X, y[..., 0]),
                              np.einsum("cn,cn->c", y[..., 0], y[..., 0])[:, None], np.full((C, 1), float(nd))], axis=1)
        terms.append(K.term(K.TERM_NORMAL_LINEAR, stats=K.vec(dv(rec), rec.shape[1]), n_data=nd,
                            scalar=K.vec(dv([tau])), transform_exp=tr))
        terms.append(K.term(K.TERM_NORMAL_RESPONSE, mat_kind=K.MAT_DENSE, P=K.vec(dv(P), p * p), scalar=K.vec(dv([lam])),
                            logdet=K.vec(dv(logdetP), 1)))
        theta0 = bt[..., 0] + 0.05 * rng.standard_normal((C, p))
        for c in range(C):
            oterms[c] = [mh.Term("normal_linear", data=y[c], X=X[c], Q=tau * np.eye(nd), transform=tr),
                         mh.Term("normal_response", p1=np.zeros((p, 1)), Q=lam * P[c])]
        return terms, keep, theta0, oterms, 0.9
    if kind == "lognormal":
        lam, tau = 50.0, 10.0
        mu = 0.2 * rng.standard_normal((C, p))
        theta0 = np.exp(mu + 0.03 * rng.standard_normal((C, p)))
        yobs = theta0 + 0.1 * rng.standard_normal((C, p))
        w = rng.uniform(0.5, 1.5, (C, p))
        terms.append(K.term(K.TERM_LOGNORMAL_RESPONSE, mat_kind=K.MAT_DENSE, p1_len=p, p1=K.vec(dv(mu), p),
                            P=K.vec(dv(P), p * p), scalar=K.vec(dv([lam])), logdet=K.vec(dv(logdetP), 1)))
        terms.append(K.term(K.TERM_NORMAL_RESPONSE, mat_kind=K.MAT_DIAG, p1_len=p, p1=K.vec(dv(yobs), p),
                            P=K.vec(dv(w), p), scalar=K.vec(dv([tau])), logdet=K.vec(dv(np.log(w).sum(1)), 1)))
        for c in range(C):
            oterms[c] = [mh.Term("lognormal_response", p1=mu[c].reshape(-1, 1), Q=lam * P[c]),
                         mh.Term("normal_response", p1=yobs[c].reshape(-1, 1), Q=tau * np.diag(w[c]))]
        return terms, keep, theta0, oterms, 0.5
    if kind == "poisson":
        lam = 0.5
        mu0 = np.full((C, p), 20.0)
        k = rng.poisson(20.0, (C, p)).astype(float)
        theta0 = 20.0 + rng.standard_normal((C, p))
        terms.append(K.term(K.TERM_POISSON_RATE, data=K.vec(dv(k), p)))
        terms.append(K.term(K.TERM_NORMAL_RESPONSE, mat_kind=K.MAT_DENSE, p1_len=p, p1=K.vec(dv(mu0), p),
                            P=K.vec(dv(P), p * p), scalar=K.vec(dv([lam])), logdet=K.vec(dv(logdetP), 1)))
        for c in range(C):
            oterms[c] = [mh.Term("poisson_rate", data=k[c].reshape(-1, 1)),
                         mh.Term("normal_response", p1=mu0[c].reshape(-1, 1), Q=lam * P[c])]
        return terms, keep, theta0, oterms, 0.8
    raise ValueError(kind)


def _elem_case(kind, n, C, seed):
    """Per-chain data for one element-wise model (Poisson-Gamma or a diagonal Normal prior + diagonal observation)."""
    from openmcmc_b200 import kernels as K
    from oracle import mh

    rng = np.random.default_rng(seed)
    keep, oterms = [], [[] for _ in range(C)]

    def dv(x):
        t = _dev(x)
        keep.append(t)
        return t

    if kind == "poisson_gamma":
        a, b = rng.uniform(2.0, 4.0, (C, n)), rng.uniform(0.5, 1.5, (C, n))
        k = rng.poisson(5.0, (C, n)).astype(float)
        theta0 = (k + a) / (b + 1.0) * rng.uniform(0.8, 1.2, (C, n))
        terms = [K.term(K.TERM_POISSON_RATE, data=K.vec(dv(k), n)),
                 K.term(K.TERM_GAMMA_RESPONSE, p1_len=n, p2_len=n, p1=K.vec(dv(a), n), p2=K.vec(dv(b), n))]
        for c in range(C):
            oterms[c] = [mh.Term("poisson_rate", data=k[c].reshape(-1, 1)),
                         mh.Term("gamma_response", p1=a[c].reshape(-1, 1), p2=b[c].reshape(-1, 1))]
        return terms, keep, theta0, oterms, 0.9
    m, w, yobs, v = (rng.standard_normal((C, n)), rng.uniform(0.5, 2.0, (C, n)), rng.standard_normal((C, n)),
                     rng.uniform(0.5, 2.0, (C, n)))
    lam, tau = 2.0, 3.0
    theta0 = rng.standard_normal((C, n))
    terms = [K.term(K.TERM_NORMAL_RESPONSE, mat_kind=K.MAT_DIAG, p1_len=n, p1=K.vec(dv(m), n), P=K.vec(dv(w), n),
                    scalar=K.vec(dv([lam])), logdet=K.vec(dv(np.log(w).sum(1)), 1)),
             K.term(K.TERM_NORMAL_RESPONSE, mat_kind=K.MAT_DIAG, p1_len=n, p1=K.vec(dv(yobs), n), P=K.vec(dv(v), n),
                    scalar=K.vec(dv([tau])), logdet=K.vec(dv(np.log(v).sum(1)), 1))]
    for c in range(C):
        oterms[c] = [mh.Term("normal_response", p1=m[c].reshape(-1, 1), Q=lam * np.diag(w[c])),
                     mh.Term("normal_response", p1=yobs[c].reshape(-1, 1), Q=tau * np.diag(v[c]))]
    return terms, keep, theta0, oterms, 0.9


def _workspace(C, n):
    import torch

    from openmcmc_b200 import kernels as K

    ws = K.nn_dense_workspace(C, n)
    return torch.empty(ws, dtype=torch.float64, device="cuda") if ws > 0 else None


def _replay(terms, theta0, oterms, step, n_steps, seed, check_probes=True):
    """Runs the kernel step by step with injected z / u and probes, and the oracle chain by chain beside it."""
    import torch

    from openmcmc_b200 import kernels as K
    from oracle import mh

    C, n = theta0.shape
    rng = np.random.default_rng(seed + 1)
    model = K.mh_model(C, n, terms)
    theta = _dev(theta0)
    ws = _workspace(C, n)
    status = torch.zeros(C, dtype=torch.int32, device="cuda")
    counters = torch.zeros(C, 2, dtype=torch.int64, device="cuda")
    pmu, pprop, psc = (torch.zeros(C, n, dtype=torch.float64, device="cuda"),
                       torch.zeros(C, n, dtype=torch.float64, device="cuda"),
                       torch.zeros(C, 6, dtype=torch.float64, device="cuda"))
    pL = torch.zeros(C, n, n, dtype=torch.float64, device="cuda") if check_probes else None
    th = [theta0[c].reshape(-1, 1).copy() for c in range(C)]
    n_acc = np.zeros(C, dtype=int)
    for it in range(n_steps):
        z, u = rng.standard_normal((C, n)), rng.uniform(size=C)
        K.mmala(model, theta, step, 0, K.rng(seed), debug_z=_dev(z), debug_u=_dev(u), counters=counters, status=status,
                probe_mu=pmu, probe_L=pL, probe_prop=pprop, probe_scalars=psc, workspace=ws)
        torch.cuda.synchronize()
        got, gmu, gprop, gsc = theta.cpu().numpy(), pmu.cpu().numpy(), pprop.cpu().numpy(), psc.cpu().numpy()
        gL = pL.cpu().numpy() if check_probes else None
        gst = status.cpu().numpy()
        for c in range(C):
            try:
                th_new, info = mh.mmala_step(oterms[c], th[c], step, z[c], u[c], "analytic")
            except np.linalg.LinAlgError:       # not PD at the current point: rejected and flagged, no proposal
                assert gst[c] & 1 and gsc[c, 5] == 0.0
                np.testing.assert_array_equal(got[c], th[c].ravel())
                continue
            th[c] = th_new
            np.testing.assert_allclose(gmu[c], info["mu"].ravel(), rtol=1e-10, atol=1e-12 * np.abs(info["mu"]).max())
            np.testing.assert_allclose(gprop[c], info["prop"].ravel(), rtol=1e-9, atol=1e-11 * np.abs(info["prop"]).max())
            if check_probes:
                np.testing.assert_allclose(gL[c], info["L"], rtol=1e-10, atol=1e-12 * np.abs(info["L"]).max())
            if info["invalid"]:
                assert gsc[c, 5] == 0.0
            else:
                want = np.array([info["logp_cur"], info["logp_prop"], info["lq_fwd"], info["lq_rev"],
                                 info["log_accept"]])
                fin = np.isfinite(want)
                np.testing.assert_allclose(gsc[c, :5][fin], want[fin], rtol=1e-9)
                # a proposal outside the support: the device's Poisson term is NaN at a negative rate (scipy's
                # convention, as in every MH kernel), the oracle's -inf where the count is 0; both reject
                assert not np.any(np.isfinite(gsc[c, :5][~fin]))
                assert bool(gsc[c, 5]) == info["accepted"], (it, c)
            n_acc[c] += info["accepted"]
            np.testing.assert_allclose(got[c], th[c].ravel(), rtol=1e-9, atol=1e-12)
    assert np.array_equal(counters.cpu().numpy()[:, 0], n_acc)
    assert np.array_equal(counters.cpu().numpy()[:, 1], np.full(C, n_steps))
    return n_acc


# ------------------------------------------------------------------------------------------------ 1. dense vs oracle
DENSE_P = [65, 72, 80, 128, 136, 137, 200, 511, 512]


@pytest.mark.parametrize("kind", ["linear", "linear_exp", "lognormal", "poisson"])
@pytest.mark.parametrize("p", DENSE_P)
def test_dense_step_matches_oracle(kind, p):
    from openmcmc_b200 import kernels as K

    K.init_device()
    C, steps = (64, 10) if p <= 137 else ((8, 6) if p <= 200 else (4, 3))
    terms, keep, theta0, oterms, step = _dense_case(kind, p, C, seed=p)
    _replay(terms, theta0, oterms, step, n_steps=steps, seed=p)


# ------------------------------------------------------------------------------------------------ 2. element-wise
@pytest.mark.parametrize("kind", ["poisson_gamma", "normal_diag"])
@pytest.mark.parametrize("n", [65, 100, 1000, 4096])
def test_elementwise_step_matches_oracle(kind, n):
    from openmcmc_b200 import kernels as K

    K.init_device()
    C = {65: 64, 100: 64, 1000: 6, 4096: 2}[n]
    terms, keep, theta0, oterms, _ = _elem_case(kind, n, C, seed=n)
    step = n ** (-1.0 / 6.0)     # Langevin acceptance falls with the dimension unless the step shrinks like n^(-1/6)
    _replay(terms, theta0, oterms, step, n_steps=10 if n <= 1000 else 3, seed=n, check_probes=n <= 1000)


# ------------------------------------------------------------------------------------------------ 3. through MCMC
def _reg_model_state(p, seed, transform=True, nd=None):
    from openmcmc_b200.distribution.location_scale import Normal
    from openmcmc_b200.model import Model
    from openmcmc_b200.parameter import LinearCombination, LinearCombinationWithTransform, ScaledMatrix
    from oracle import mh

    rng = np.random.default_rng(seed)
    nd = nd or 2 * p
    X = rng.standard_normal((nd, p)) / np.sqrt(p)
    bt = 0.1 * rng.standard_normal((p, 1))
    y = X @ (np.exp(bt) if transform else bt) + 0.2 * rng.standard_normal((nd, 1))
    P = _spd(rng, p)
    tau, lam = 4.0, 1.0
    mean = (LinearCombinationWithTransform(form={"beta": "X"}, transform={"beta": True}) if transform
            else LinearCombination(form={"beta": "X"}))
    mdl = Model([Normal("y", mean=mean, precision=ScaledMatrix(matrix="W", scalar="tau")),
                 Normal("beta", mean="mu", precision=ScaledMatrix(matrix="P", scalar="lam"))])
    state = {"y": y, "X": X, "beta": bt + 0.05 * rng.standard_normal((p, 1)), "W": sparse.identity(nd, format="csc"),
             "tau": tau, "mu": np.zeros((p, 1)), "P": P, "lam": lam}
    terms = [mh.Term("normal_linear", data=y, X=X, Q=tau * np.eye(nd), transform=transform),
             mh.Term("normal_response", p1=np.zeros((p, 1)), Q=lam * P)]
    return mdl, state, terms


@pytest.mark.parametrize("p", [80, 200])
def test_mmala_regression_through_mcmc(p):
    from openmcmc_b200.mcmc import MCMC
    from openmcmc_b200.sampler.metropolis_hastings import ManifoldMALA
    from oracle import mh

    mdl, state, terms = _reg_model_state(p, seed=p)
    n_iter, step = 8, 0.9
    rng = np.random.default_rng(7)
    z, u = rng.standard_normal((n_iter, p)), rng.uniform(size=n_iter)
    beta0 = state["beta"].copy()
    smp = ManifoldMALA("beta", mdl, step=np.array([[step]]))
    M = MCMC(state, [smp], model=mdl, n_burn=0, n_iter=n_iter, debug_draws={"beta": {"z": z, "u": u}})
    M.run_mcmc()
    theta, n_acc = beta0, 0
    for it in range(n_iter):
        theta, info = mh.mmala_step(terms, theta, step, z[it], u[it], "analytic")
        n_acc += info["accepted"]
        np.testing.assert_allclose(M.store["beta"][:, it], theta.ravel(), rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(M.store["log_post"][it, 0], mh.log_p(terms, theta), rtol=1e-10)
    assert smp.accept_rate.count == {"accept": n_acc, "proposal": n_iter}


def test_grad_log_p_and_random_walk_at_p200():
    from openmcmc_b200.mcmc import MCMC
    from openmcmc_b200.sampler.metropolis_hastings import RandomWalk
    from oracle import mh

    p = 200
    mdl, state, terms = _reg_model_state(p, seed=3)
    gr, H = mdl["y"].grad_log_p(state, "beta", hessian_required=True)
    go, Ho = terms[0].grad_hess_analytic(state["beta"])
    np.testing.assert_allclose(gr, go, rtol=1e-9, atol=1e-10 * np.abs(go).max())
    np.testing.assert_allclose(H, Ho, rtol=1e-10, atol=1e-12 * np.abs(Ho).max())
    np.testing.assert_allclose(mdl["y"].log_p(state), terms[0].log_p(state["beta"]), rtol=1e-10)
    n_iter, step = 8, np.array([[0.01]])
    rng = np.random.default_rng(5)
    z, u = rng.standard_normal((n_iter, p)), rng.uniform(size=n_iter)
    theta = state["beta"].copy()
    M = MCMC(state, [RandomWalk("beta", mdl, step=step)], model=mdl, n_burn=0, n_iter=n_iter,
             debug_draws={"beta": {"z": z, "u": u}})
    M.run_mcmc()
    for it in range(n_iter):
        theta, info = mh.random_walk_step(terms, theta, step, z[it].reshape(theta.shape), u[it], None)
        np.testing.assert_allclose(M.store["beta"][:, it], theta.ravel(), rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(M.store["log_post"][it, 0], mh.log_p(terms, theta), rtol=1e-10)


# ------------------------------------------------------------------------------------------------ 4. free running
def test_dense_free_running_matches_conjugate_posterior():
    from openmcmc_b200.mcmc import MCMC
    from openmcmc_b200.sampler.metropolis_hastings import ManifoldMALA

    p = 100
    mdl, state, _ = _reg_model_state(p, seed=11, transform=False)
    C = 1024
    # the step shrinks like p^(-1/6) (0.6 accepts almost nothing at p = 100); one draw per chain after burn-in
    smp = ManifoldMALA("beta", mdl, step=np.array([[0.25]]))
    M = MCMC(state, [smp], model=mdl, n_burn=600, n_iter=1, n_chains=C, seed=2)
    M.run_mcmc()
    b = M.store["beta"]                                                  # (C, p, n_iter)
    X, y = state["X"], state["y"]
    Q = state["tau"] * X.T @ X + state["lam"] * state["P"]
    mean = np.linalg.solve(Q, state["tau"] * X.T @ y).ravel()
    sd = np.sqrt(np.diag(np.linalg.inv(Q)))
    draws = b[:, :, -1].T                                                # (p, C)
    se = sd / np.sqrt(C)
    assert np.all(np.abs(draws.mean(axis=1) - mean) < 5 * se), np.abs(draws.mean(axis=1) - mean) / se
    assert np.all(np.abs(draws.std(axis=1) / sd - 1) < 0.2)


def test_elementwise_free_running_poisson_gamma_posterior():
    from openmcmc_b200.distribution.distribution import Gamma, Poisson
    from openmcmc_b200.mcmc import MCMC
    from openmcmc_b200.model import Model
    from openmcmc_b200.sampler.metropolis_hastings import ManifoldMALA

    n, C = 256, 1024
    rng = np.random.default_rng(4)
    y = rng.poisson(6.0, (n, 1)).astype(float)
    a, b = 3.0, 1.0
    mdl = Model([Poisson("y", rate="lam"), Gamma("lam", shape="a", rate="b")])
    # started at the posterior means: a Langevin chain with 256 coordinates started in the tail of some of them rejects
    # nearly every joint move; the step is small for the same reason (n = 64 at step 0.5 accepts ~2 % of the moves)
    state = {"y": y, "lam": (a + y) / (b + 1.0), "a": a, "b": b}
    smp = ManifoldMALA("lam", mdl, step=np.array([[0.15]]))
    M = MCMC(state, [smp], model=mdl, n_burn=2000, n_iter=1, n_chains=C, seed=9)
    M.run_mcmc()
    last = M.store["lam"][:, :, -1]                                      # (C, n)
    pvals = np.array([stats.kstest(last[:, j], stats.gamma(a + y[j, 0], scale=1.0 / (b + 1.0)).cdf).pvalue
                      for j in range(n)])
    assert 5 < smp.accept_rate.acceptance_rate < 99.9, smp.accept_rate.acceptance_rate
    assert pvals.min() > 1e-3 / n, pvals.min()


# ------------------------------------------------------------------------------------------------ 5. invariance, failure
@pytest.mark.parametrize("kind,n", [("dense", 137), ("elem", 300)])
def test_chain_slice_matches_full_launch(kind, n):
    import torch

    from openmcmc_b200 import _cabi
    from openmcmc_b200 import kernels as K

    K.init_device()
    C, h = 32, 16
    terms, keep, theta0, _, step = (_dense_case("poisson", n, C, seed=1) if kind == "dense"
                                    else _elem_case("poisson_gamma", n, C, seed=1))
    step = min(step, 0.1 if kind == "elem" else 0.5)   # small enough that some of the joint moves are accepted

    def run(chains, offset):
        sub = []
        for t in terms:        # the same operands seen from chain `offset` on
            t2 = K.term(t.kind, t.mat_kind, t.p1_len, t.p2_len)
            for f in ("data", "p1", "p2", "P", "scalar", "logdet", "stats"):
                v = getattr(t, f)
                ptr = (v.ptr or 0) + 8 * offset * v.chain_stride if v.ptr else None
                setattr(t2, f, _cabi.Vec(ptr, v.chain_stride))
            t2.dom_lo, t2.dom_hi, t2.n_data, t2.transform_exp = t.dom_lo, t.dom_hi, t.n_data, t.transform_exp
            sub.append(t2)
        th = _dev(theta0[offset:offset + chains])
        sweep = torch.zeros(1, dtype=torch.int64, device="cuda")
        for s in range(3):
            sweep.fill_(s)
            K.mmala(K.mh_model(chains, n, sub), th, step, 0, K.rng(21, sweep=sweep, chain_offset=offset),
                    workspace=_workspace(chains, n))
        return th.cpu().numpy()

    full = run(C, 0)
    part = run(C - h, h)
    np.testing.assert_array_equal(part, full[h:])
    assert not np.array_equal(full, theta0)


@pytest.mark.parametrize("kind,n", [("dense", 96), ("dense", 200), ("elem", 65), ("elem", 2000)])
def test_failing_chains_are_rejected_and_flagged(kind, n):
    import torch

    from openmcmc_b200 import kernels as K

    K.init_device()
    C = 8
    terms, keep, theta0, _, step = (_dense_case("poisson", n, C, seed=2) if kind == "dense"
                                    else _elem_case("poisson_gamma", n, C, seed=2))
    rng = np.random.default_rng(3)
    z, u = rng.standard_normal((C, n)), rng.uniform(size=C)

    def run(theta_init, zz):
        th = _dev(theta_init)
        status = torch.zeros(C, dtype=torch.int32, device="cuda")
        K.mmala(K.mh_model(C, n, terms), th, step, 0, K.rng(0), debug_z=_dev(zz), debug_u=_dev(u), status=status,
                workspace=_workspace(C, n))
        return th.cpu().numpy(), status.cpu().numpy()

    ref, st_ref = run(theta0, z)
    bad = theta0.copy()
    bad[1] = -np.abs(bad[1])      # negative rates: the Poisson Hessian k / x^2 stays positive but the gradient and
    bad[1, 0] = 0.0               # log-density are not finite at x = 0 -> NOT_PD (rejected before any proposal)
    zz = z.copy()
    zz[5] = -50.0                 # drives every coordinate of chain 5 far below zero: invalid proposal
    got, st = run(bad, zz)
    np.testing.assert_array_equal(got[1], bad[1])
    np.testing.assert_array_equal(got[5], theta0[5])
    assert st[1] == 1 and st[5] == 4, st
    others = [c for c in range(C) if c not in (1, 5)]
    np.testing.assert_array_equal(got[others], ref[others])
    np.testing.assert_array_equal(st[others], st_ref[others])


# ------------------------------------------------------------------------------------------------ 6. refusals
def test_refusals():
    import torch

    from openmcmc_b200 import _cabi, engine
    from openmcmc_b200 import kernels as K
    from openmcmc_b200.distribution.distribution import Gamma, Poisson
    from openmcmc_b200.mcmc import MCMC
    from openmcmc_b200.model import Model
    from openmcmc_b200.sampler.metropolis_hastings import ManifoldMALA

    K.init_device()
    mdl, state, _ = _reg_model_state(513, seed=0, transform=False, nd=600)
    with pytest.raises(engine.PlanError, match="513 > 512"):
        MCMC(state, [ManifoldMALA("beta", mdl, step=np.array([[0.5]]))], model=mdl, n_burn=0, n_iter=1).run_mcmc()
    pg = Model([Poisson("y", rate="lam"), Gamma("lam", shape="a", rate="b")])
    for n, deriv, msg in ((4097, "analytic", "4097 > 4096"), (65, "fd", "derivatives='fd'")):
        st = {"y": np.ones((n, 1)), "lam": np.ones((n, 1)), "a": 2.0, "b": 1.0}
        with pytest.raises(engine.PlanError, match=msg):
            MCMC(st, [ManifoldMALA("lam", pg, step=np.array([[0.5]]), derivatives=deriv)], model=pg, n_burn=0,
                 n_iter=1).run_mcmc()
    # the C entry point refuses the same on its own
    for kind, n in (("dense", 513), ("elem", 4097)):
        C = 2
        if kind == "dense":
            P = _dev(np.eye(n))
            terms = [K.term(K.TERM_NORMAL_RESPONSE, mat_kind=K.MAT_DENSE, P=K.vec(P))]
        else:
            k = _dev(np.ones(n))
            terms = [K.term(K.TERM_POISSON_RATE, data=K.vec(k))]
        th = torch.ones(C, n, dtype=torch.float64, device="cuda")
        with pytest.raises(_cabi.OmcError):
            K.mmala(K.mh_model(C, n, terms), th, 0.5, 0, K.rng(0))
    k = _dev(np.ones(65))
    with pytest.raises(_cabi.OmcError):
        K.mmala(K.mh_model(2, 65, [K.term(K.TERM_POISSON_RATE, data=K.vec(k))]),
                torch.ones(2, 65, dtype=torch.float64, device="cuda"), 0.5, 1, K.rng(0))
