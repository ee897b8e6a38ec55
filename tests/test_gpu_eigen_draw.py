"""The dense NormalNormal draw in a fixed eigenbasis (omc_nn_eigen_prep / omc_nn_eigen_draw, p <= 64).

The prep factors M'P0M = I, M'GM = D once per chain; a sweep's draw is then beta = M u with u element-wise.  Checked
here at p = 1 ... 64 with P0 the identity, a scaled identity and a positive diagonal, cond(G) from 1 to 1e12, a
rank-deficient G and one with repeated eigenvalues:

* the prep against torch fp64: P0 M D M' P0 = G and M'P0M = I to a few p eps;
* z = 0: the mean against torch.linalg.solve(Q, b) within c eps cond(Q);
* z = e_i: the square root A = M S^-1/2 satisfies A'QA = I;
* free-running Philox with the Cholesky kernel's RNG site: (beta - mu)'Q(beta - mu) is the same z'z for both kernels;
* rss = rss0 - 2 d'c0 + d'G d against a long-double evaluation at the returned beta;
* a KS test of whitened draws; bit-identical repeats and chain_offset shards; failing chains flagged alone;
* the plan: the eigen path on the C2 model, the Cholesky path with injected draws, a truncated prior and p = 80.
"""

import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PS = [1, 3, 8, 33, 41, 57, 63, 64]
PRIORS = ["eye", "scaled", "diag"]
EPS = np.finfo(np.float64).eps


def _G(C, p, kind, g):
    """[C, p, p] symmetric PSD test matrices: cond(G) = kind (a number), 'rank' (X'X with n = p/2 rows) or 'repeat'
    (eigenvalues 1 and 3, each about p/2 times)."""
    import torch

    dev, f64 = "cuda", torch.float64
    if kind == "rank":
        X = torch.randn(C, max(p // 2, 1), p, dtype=f64, device=dev, generator=g)
        G = X.transpose(1, 2) @ X
    else:
        U, _ = torch.linalg.qr(torch.randn(C, p, p, dtype=f64, device=dev, generator=g))
        if kind == "repeat":
            ev = torch.where(torch.arange(p, device=dev) % 2 == 0, 1.0, 3.0).to(f64)
        else:
            ev = torch.logspace(0.0, -math.log10(kind), p, dtype=f64, device=dev)
        G = (U * ev) @ U.transpose(1, 2)
    return 0.5 * (G + G.transpose(1, 2))


def _problem(C, p, prior, gkind, seed, lam=None, same=False):
    import torch

    from openmcmc_b200 import kernels as K

    dev, f64 = "cuda", torch.float64
    g = torch.Generator(device=dev).manual_seed(seed)
    G = _G(1 if same else C, p, gkind, g).expand(C, p, p).contiguous()
    gv = torch.randn(1 if same else C, p, dtype=f64, device=dev, generator=g).expand(C, p).contiguous()
    stats = torch.cat([G.reshape(C, -1), gv, torch.zeros(C, 2, dtype=f64, device=dev)], dim=1).contiguous()
    if prior == "eye":
        pd, kind, Pv = torch.ones(p, dtype=f64, device=dev), K.MAT_EYE, None
    elif prior == "scaled":
        Pv = torch.full((1,), 2.5, dtype=f64, device=dev)
        pd, kind = Pv.expand(p), K.MAT_EYE
    else:
        Pv = torch.rand(p, dtype=f64, device=dev, generator=g) * 4.0 + 0.25
        pd, kind = Pv, K.MAT_DIAG
    mu0 = torch.randn(p, dtype=f64, device=dev, generator=g)
    tau = torch.rand(C, dtype=f64, device=dev, generator=g) + 0.5
    lam = (torch.rand(C, dtype=f64, device=dev, generator=g) + 0.5) * (1e-3 if lam is None else lam)
    bhat = torch.randn(C, p, dtype=f64, device=dev, generator=g)
    c0 = torch.randn(C, p, dtype=f64, device=dev, generator=g)
    rss0 = torch.rand(C, 1, dtype=f64, device=dev, generator=g) * 100.0 + 1.0
    center = torch.cat([bhat, c0, rss0, torch.zeros(C, 1, dtype=f64, device=dev)], dim=1).contiguous()
    Q = lam.view(-1, 1, 1) * torch.diag(pd) + tau.view(-1, 1, 1) * G
    b = lam.view(-1, 1) * pd * mu0 + tau.view(-1, 1) * gv
    return dict(C=C, p=p, G=G, gv=gv, stats=stats, kind=kind, Pv=Pv, pd=pd, mu0=mu0, tau=tau, lam=lam, center=center,
                Q=Q, b=b)


def _prep(pr):
    import torch

    from openmcmc_b200 import kernels as K

    C, p = pr["C"], pr["p"]
    eig = torch.zeros(C, K.eigen_record_len(p), dtype=torch.float64, device="cuda")
    K.nn_eigen_prep(C, p, pr["stats"], pr["kind"], K.vec(pr["Pv"]), K.vec(pr["mu0"]), pr["center"], eig)
    return eig


def _draw(pr, eig, z=None, rng=None, chains=None, status_ok=True):
    import torch

    from openmcmc_b200 import kernels as K

    p = pr["p"]
    sl = slice(0, pr["C"]) if chains is None else chains
    n = sl.stop - sl.start
    rss = torch.zeros(n, dtype=torch.float64, device="cuda")
    beta = torch.empty(n, p, dtype=torch.float64, device="cuda")
    status = torch.zeros(n, dtype=torch.int32, device="cuda")
    K.nn_eigen_draw(n, p, eig[sl].contiguous(), K.vec(pr["tau"][sl].contiguous(), 1),
                    K.vec(pr["lam"][sl].contiguous(), 1), beta, rng if rng is not None else K.rng(seed=5, site=1),
                    status=status, debug_z=None if z is None else z[sl].contiguous(),
                    center=pr["center"][sl].contiguous(), rss_out=rss.data_ptr(), rss_stride=1)
    torch.cuda.synchronize()
    if status_ok:
        assert int(status.count_nonzero()) == 0
    return beta, rss, status


def _chol_draw(pr, rng):
    import torch

    from openmcmc_b200 import kernels as K

    C, p = pr["C"], pr["p"]
    beta = torch.empty(C, p, dtype=torch.float64, device="cuda")
    K.nn_dense_draw(C, p, pr["stats"].clone(), K.vec(pr["tau"], 1), pr["kind"], K.vec(pr["Pv"]), K.vec(pr["lam"], 1),
                    K.vec(pr["mu0"]), beta, rng)
    torch.cuda.synchronize()
    return beta


def _split(eig, p):
    C = eig.shape[0]
    M = eig[:, :p * p].reshape(C, p, p).transpose(1, 2)    # column-major on the device
    v = eig[:, p * p:].reshape(C, 5, p)
    return M, v[:, 0], v[:, 1], v[:, 2], v[:, 3], v[:, 4]


@pytest.mark.parametrize("prior", PRIORS)
@pytest.mark.parametrize("p", PS)
def test_prep_factors_G_and_P0(p, prior):
    import torch

    from openmcmc_b200 import kernels as K

    K.init_device(0)
    for gkind in (1.0, 1e6, 1e12, "rank", "repeat"):
        pr = _problem(64, p, prior, gkind, seed=11 * p + len(prior))
        eig = _prep(pr)
        M, D, h, m, uh, k = _split(eig, p)
        assert bool(torch.isfinite(eig).all()), gkind
        P0 = torch.diag(pr["pd"])
        I = torch.eye(p, dtype=torch.float64, device="cuda")
        G = pr["G"]
        rec = P0 @ (M * D.unsqueeze(1)) @ M.transpose(1, 2) @ P0
        gn = torch.linalg.matrix_norm(G, ord=2).clamp_min(1e-300)
        err_g = (torch.linalg.matrix_norm(rec - G, ord=2) / gn).max().item()
        err_i = torch.linalg.matrix_norm(M.transpose(1, 2) @ P0 @ M - I, ord=2).max().item()
        assert err_g <= 4 * p * EPS and err_i <= 4 * p * EPS, (gkind, err_g / (p * EPS), err_i / (p * EPS))
        # the vectors: h = M'g, m = M'P0 mu0, u_hat = M'P0 beta_hat, k = M'c0
        Mt = M.transpose(1, 2)
        cen = pr["center"]
        for got, ref in ((h, Mt @ pr["gv"].unsqueeze(-1)), (m, Mt @ (pr["pd"] * pr["mu0"]).unsqueeze(-1).expand(64, p, 1)),
                         (uh, Mt @ (pr["pd"] * cen[:, :p]).unsqueeze(-1)), (k, Mt @ cen[:, p:2 * p].unsqueeze(-1))):
            ref = ref.squeeze(-1)
            assert bool(((got - ref).abs().amax(1) <= 8 * p * EPS * ref.abs().amax(1).clamp_min(1.0) *
                         M.abs().amax((1, 2)).clamp_min(1.0)).all()), gkind


@pytest.mark.parametrize("prior", PRIORS)
@pytest.mark.parametrize("p", PS)
def test_mean_matches_solve(p, prior):
    import torch

    from openmcmc_b200 import kernels as K

    K.init_device(0)
    for gkind in (1.0, 1e6, 1e12, "rank", "repeat"):
        pr = _problem(128, p, prior, gkind, seed=7 * p + len(prior))
        eig = _prep(pr)
        beta, _, _ = _draw(pr, eig, z=torch.zeros(128, p, dtype=torch.float64, device="cuda"))
        ref = torch.linalg.solve(pr["Q"], pr["b"].unsqueeze(-1)).squeeze(-1)
        kappa = torch.linalg.cond(pr["Q"])
        rel = (beta - ref).abs().amax(dim=1) / ref.abs().amax(dim=1)
        assert bool((rel <= 4 * p * EPS * kappa).all()), (gkind, float((rel / (EPS * kappa)).max()))


@pytest.mark.parametrize("prior", PRIORS)
@pytest.mark.parametrize("p", PS)
def test_square_root_of_the_covariance(p, prior):
    """With z = e_i the draw moves by column i of A = M S^-1/2: A'QA = I."""
    import torch

    from openmcmc_b200 import kernels as K

    K.init_device(0)
    C = 16
    pr = _problem(C, p, prior, 1e4, seed=3 * p + len(prior))
    eig = _prep(pr)
    zero = torch.zeros(C, p, dtype=torch.float64, device="cuda")
    mu, _, _ = _draw(pr, eig, z=zero)
    cols = []
    for i in range(p):
        z = zero.clone()
        z[:, i] = 1.0
        cols.append(_draw(pr, eig, z=z)[0] - mu)
    A = torch.stack(cols, dim=2)
    I = torch.eye(p, dtype=torch.float64, device="cuda")
    err = (A.transpose(1, 2) @ pr["Q"] @ A - I).abs().amax((1, 2))
    kappa = torch.linalg.cond(pr["Q"])
    assert bool((err <= 4 * p * EPS * kappa).all()), float((err / (EPS * kappa)).max())


@pytest.mark.parametrize("prior", PRIORS)
@pytest.mark.parametrize("p", [3, 8, 33, 57, 64])
def test_free_running_is_the_same_z_through_another_square_root(p, prior):
    """Same seed and site as the Cholesky kernel: both draws whiten to the same z'z."""
    import torch

    from openmcmc_b200 import kernels as K

    K.init_device(0)
    C = 512
    pr = _problem(C, p, prior, 1e3, seed=5 * p + len(prior))
    eig = _prep(pr)
    rng = K.rng(seed=21, site=3)
    be, _, _ = _draw(pr, eig, rng=rng)
    bc = _chol_draw(pr, rng)
    mu = torch.linalg.solve(pr["Q"], pr["b"].unsqueeze(-1))
    qe = ((be.unsqueeze(-1) - mu).transpose(1, 2) @ pr["Q"] @ (be.unsqueeze(-1) - mu)).flatten()
    qc = ((bc.unsqueeze(-1) - mu).transpose(1, 2) @ pr["Q"] @ (bc.unsqueeze(-1) - mu)).flatten()
    rel = ((qe - qc).abs() / qc.clamp_min(1e-300)).max().item()
    assert rel <= 1e-9, rel
    assert not bool(torch.equal(be, bc)) or p == 1


@pytest.mark.parametrize("prior", PRIORS)
@pytest.mark.parametrize("p", PS)
def test_rss_matches_long_double(p, prior):
    import torch

    from openmcmc_b200 import kernels as K

    K.init_device(0)
    C = 200
    pr = _problem(C, p, prior, 1e4, seed=17 + p + len(prior), lam=1.0)
    eig = _prep(pr)
    beta, rss, _ = _draw(pr, eig, z=torch.randn(C, p, dtype=torch.float64, device="cuda"))
    ld = np.longdouble
    b = beta.cpu().numpy().astype(ld)
    cen = pr["center"].cpu().numpy().astype(ld)
    G = pr["G"].cpu().numpy().astype(ld)
    d = b - cen[:, :p]
    c0, rss0 = cen[:, p:2 * p], cen[:, 2 * p]
    ref = rss0 - 2 * np.einsum("ci,ci->c", d, c0) + np.einsum("ci,cij,cj->c", d, G, d)
    # terms of the sum, with |beta_hat| standing in for d where the eigenbasis carries beta_hat's rounding
    ad = np.abs(d) + np.abs(cen[:, :p])
    terms = np.abs(rss0) + 2 * np.einsum("ci,ci->c", ad, np.abs(c0)) + np.einsum("ci,cij,cj->c", ad, np.abs(G), ad)
    err = np.abs(rss.cpu().numpy().astype(ld) - ref)
    assert bool(np.all(err <= 8 * p * EPS * terms)), float(np.max(err / terms))


@pytest.mark.parametrize("p", [8, 33, 64])
def test_whitened_draws_are_standard_normal(p):
    """One problem in every chain, lambda and tau fixed: L'(beta - mu) over all chains is iid N(0, 1)."""
    import torch
    from scipy import stats

    from openmcmc_b200 import kernels as K

    K.init_device(0)
    C = 4096
    pr = _problem(C, p, "diag", 1e3, seed=41 + p, same=True)
    pr["tau"].fill_(1.3)
    pr["lam"].fill_(0.2)
    pr["Q"] = pr["lam"].view(-1, 1, 1) * torch.diag(pr["pd"]) + pr["tau"].view(-1, 1, 1) * pr["G"]
    pr["b"] = pr["lam"].view(-1, 1) * pr["pd"] * pr["mu0"] + pr["tau"].view(-1, 1) * pr["gv"]
    eig = _prep(pr)
    beta, _, _ = _draw(pr, eig, rng=K.rng(seed=77, site=4))
    Q, b = pr["Q"][0], pr["b"][0]
    mu = torch.linalg.solve(Q, b)
    L = torch.linalg.cholesky(Q)
    w = ((beta - mu) @ L).cpu().numpy()          # rows: L'(beta - mu)
    assert stats.kstest(w.ravel(), "norm").pvalue > 1e-3
    cov = np.cov(w, rowvar=False)
    assert np.abs(cov - np.eye(p)).max() < 8.0 / math.sqrt(C)


@pytest.mark.parametrize("p", [3, 41, 64])
def test_repeat_and_chain_offset_shard_are_bit_identical(p):
    from openmcmc_b200 import kernels as K

    K.init_device(0)
    C, lo, hi = 4096, 1500, 2700
    pr = _problem(C, p, "diag", 1e3, seed=13 + p)
    eig = _prep(pr)
    eig2 = _prep(pr)
    assert bool((eig == eig2).all())
    b1, r1, _ = _draw(pr, eig, rng=K.rng(seed=9, site=2))
    b2, r2, _ = _draw(pr, eig, rng=K.rng(seed=9, site=2))
    assert bool((b1 == b2).all()) and bool((r1 == r2).all())
    bs, rs, _ = _draw(pr, eig, rng=K.rng(seed=9, chain_offset=lo, site=2), chains=slice(lo, hi))
    assert bool((b1[lo:hi] == bs).all()) and bool((r1[lo:hi] == rs).all())


@pytest.mark.parametrize("p", [3, 64])
def test_failing_chains_are_flagged_alone(p):
    import torch

    from openmcmc_b200 import kernels as K

    K.init_device(0)
    C = 64
    pr = _problem(C, p, "eye", 1e3, seed=19 + p)
    pr["stats"][5, 0] = float("nan")        # non-finite record: the prep marks the chain
    pr["lam"][9] = -10.0                    # S = lam + tau D <= 0
    pr["tau"][20] = float("inf")            # S not finite
    eig = _prep(pr)
    beta, _, status = _draw(pr, eig, rng=K.rng(seed=1, site=1), status_ok=False)
    bad = [5, 9, 20]
    st = status.cpu().numpy()
    assert all(st[c] == 1 for c in bad), st      # OMC_STATUS_NOT_PD
    assert np.count_nonzero(st) == len(bad)
    fin = torch.isfinite(beta).all(dim=1).cpu().numpy()
    assert not fin[bad].any() and fin.sum() == C - len(bad)


def _regression_mcmc(p, debug=False, trunc=False, n=120, C=3):
    from scipy import sparse

    from openmcmc_b200.distribution.distribution import Gamma
    from openmcmc_b200.distribution.location_scale import Normal
    from openmcmc_b200.mcmc import MCMC
    from openmcmc_b200.model import Model
    from openmcmc_b200.parameter import LinearCombination, ScaledMatrix
    from openmcmc_b200.sampler.sampler import NormalGamma, NormalNormal

    rng = np.random.default_rng(p)
    X = rng.standard_normal((C, n, p))
    y = X @ rng.standard_normal((C, p, 1)) + 0.1 * rng.standard_normal((C, n, 1))
    kw = {}
    if trunc:
        kw = dict(domain_response_lower=np.full((p, 1), -50.0), domain_response_upper=np.full((p, 1), 50.0))
    mdl = Model([
        Normal("y", mean=LinearCombination(form={"beta": "X"}), precision=ScaledMatrix(matrix="P_tau", scalar="tau")),
        Normal("beta", mean="mu", precision=ScaledMatrix(matrix="P_lambda", scalar="lambda"), **kw),
        Gamma("tau", shape="a", rate="b"), Gamma("lambda", shape="a", rate="b")])
    samplers = [NormalNormal("beta", mdl), NormalGamma("tau", mdl), NormalGamma("lambda", mdl)]
    state = {"y": y, "X": X, "beta": np.zeros((p, 1)), "P_tau": sparse.identity(n, format="csc"), "tau": 1.0,
             "P_lambda": sparse.identity(p, format="csc"), "mu": np.zeros((p, 1)), "lambda": 0.01, "a": 1e-3,
             "b": 1e-3}
    sweeps = 4
    dd = None
    if debug:
        dd = {"beta": {"z": rng.standard_normal((sweeps, C, p))}}
    M = MCMC(state, samplers, model=mdl, n_burn=0, n_iter=sweeps, n_chains=C, seed=2, debug_draws=dd)
    M.run_mcmc()
    return M


@pytest.mark.parametrize("case, eigen", [("c2", True), ("debug", False), ("trunc", False), ("p80", False)])
def test_plan_selects_the_eigen_path(case, eigen):
    M = _regression_mcmc(80 if case == "p80" else 16, debug=case == "debug", trunc=case == "trunc")
    pro = [label for label, _ in M._ops["prologue"]]
    sweep = [label for label, _ in M._ops["sweep"]]
    assert ("nn_eigen_prep" in pro) == eigen, pro
    assert "nn_eigen_prep" not in sweep and any(x.startswith("nn_dense_draw[beta]") for x in sweep), sweep
    beta = M.store["beta"]
    assert np.isfinite(beta).all()
