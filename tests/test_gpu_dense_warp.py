"""GPU parity of omc_nn_dense_draw's one-warp-per-chain kernels (p <= 64, no probes): the register kernel for small p,
the left-looking kernel with the factor in shared memory above it.

Every case injects z and compares against a torch fp64 restatement, Q = lam*P0 + tau*G, b = lam*P0 mu0 + tau*g,
x = L^-T (L^-1 b + z); chain counts cover one partial CTA, more than two rounds of the persistent warps, and a ragged
last round.  Also: solve-only mode with the relative ridge, a non-PD chain inside a batch, the rss epilogue against an
explicit d'Gd, and bit equality of a launch against a slice of it launched alone with the RNG's chain offset.
"""

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

EYE, DIAG, DENSE = 0, 1, 2


def _problem(C, p, kind, seed):
    import torch

    g = torch.Generator(device="cuda").manual_seed(seed)
    dev, f64 = "cuda", torch.float64
    A = torch.randn(C, 2 * p + 3, p, dtype=f64, device=dev, generator=g)
    G = A.transpose(1, 2) @ A / (2 * p + 3)
    gv = torch.randn(C, p, dtype=f64, device=dev, generator=g)
    stats = torch.cat([G.reshape(C, -1), gv, torch.zeros(C, 2, dtype=f64, device=dev)], dim=1).contiguous()
    tau = torch.rand(C, dtype=f64, device=dev, generator=g) * 2.0 + 0.5
    lam = torch.rand(C, dtype=f64, device=dev, generator=g) + 0.1
    mu0 = torch.randn(C, p, dtype=f64, device=dev, generator=g)
    if kind == EYE:
        P0 = None
        P0m = torch.eye(p, dtype=f64, device=dev).expand(C, p, p)
    elif kind == DIAG:
        P0 = torch.rand(C, p, dtype=f64, device=dev, generator=g) + 0.5
        P0m = torch.diag_embed(P0)
    else:
        B = torch.randn(C, p, p, dtype=f64, device=dev, generator=g)
        P0 = (B @ B.transpose(1, 2) / p + torch.eye(p, dtype=f64, device=dev)).contiguous()
        P0m = P0
    z = torch.randn(C, p, dtype=f64, device=dev, generator=g)
    return dict(C=C, p=p, kind=kind, G=G, gv=gv, stats=stats, tau=tau, lam=lam, mu0=mu0, P0=P0, P0m=P0m, z=z)


def _draw(pr, z=None, solve_only=False, ridge=0.0, status=None, center=None, rss_out=None, rng=None, chains=None):
    import torch

    from openmcmc_b200 import kernels as K

    C, p = pr["C"], pr["p"]
    sl = slice(None) if chains is None else chains
    n = C if chains is None else chains.stop - chains.start
    P0 = pr["P0"]
    pvec = K.vec(None) if P0 is None else K.vec(P0[sl].contiguous().view(n, -1), P0[0].numel())
    beta = torch.empty(n, p, dtype=torch.float64, device="cuda")
    ws_n = K.nn_dense_workspace(n, p)
    ws = torch.empty(ws_n, dtype=torch.float64, device="cuda") if ws_n else None
    stats = pr["stats"][sl].contiguous()
    K.nn_dense_draw(n, p, stats, K.vec(pr["tau"][sl].contiguous(), 1), pr["kind"], pvec,
                    K.vec(pr["lam"][sl].contiguous(), 1), K.vec(pr["mu0"][sl].contiguous(), p), beta,
                    rng if rng is not None else K.rng(seed=7, site=1), debug_z=z, status=status, center=center,
                    rss_out=rss_out if rss_out is None else stats.data_ptr() + 8 * (p * p + p),
                    solve_only=solve_only, ridge_rel=ridge, workspace=ws)
    torch.cuda.synchronize()
    return beta, stats


def _reference(pr, z, ridge=None):
    import torch

    Q = pr["lam"].view(-1, 1, 1) * pr["P0m"] + pr["tau"].view(-1, 1, 1) * pr["G"]
    if ridge is not None:
        Q = Q + torch.diag_embed(torch.diagonal(Q, dim1=1, dim2=2) * ridge)
    b = pr["lam"].view(-1, 1) * (pr["P0m"] @ pr["mu0"].unsqueeze(-1)).squeeze(-1) + pr["tau"].view(-1, 1) * pr["gv"]
    L = torch.linalg.cholesky(Q)
    w = torch.linalg.solve_triangular(L, b.unsqueeze(-1), upper=False)
    if z is not None:
        w = w + z.unsqueeze(-1)
    return torch.linalg.solve_triangular(L.transpose(1, 2), w, upper=True).squeeze(-1)


def _rel(x, ref):
    return float(((x - ref).abs().amax(dim=1) / ref.abs().amax(dim=1)).max())


@pytest.mark.parametrize("p", [64, 56, 63, 57, 48, 33, 8, 1])
@pytest.mark.parametrize("C", [1, 3, 4096, 5003])
def test_draw_matches_torch(p, C):
    from openmcmc_b200 import kernels as K

    K.init_device(0)
    pr = _problem(C, p, EYE, seed=1000 * p + C)
    beta, _ = _draw(pr, z=pr["z"])
    assert _rel(beta, _reference(pr, pr["z"])) <= 1e-9


@pytest.mark.parametrize("kind", [DIAG, DENSE])
@pytest.mark.parametrize("p", [64, 57, 48, 33, 8])
def test_draw_priors_match_torch(p, kind):
    from openmcmc_b200 import kernels as K

    K.init_device(0)
    pr = _problem(37, p, kind, seed=7 * p + kind)
    beta, _ = _draw(pr, z=pr["z"])
    assert _rel(beta, _reference(pr, pr["z"])) <= 1e-9


@pytest.mark.parametrize("p", [64, 63, 48, 8])
def test_solve_only_with_ridge(p):
    from openmcmc_b200 import kernels as K

    K.init_device(0)
    pr = _problem(300, p, EYE, seed=p)
    beta, _ = _draw(pr, solve_only=True, ridge=1e-6)
    assert _rel(beta, _reference(pr, None, ridge=1e-6)) <= 1e-9


@pytest.mark.parametrize("p", [64, 57, 8])
def test_non_pd_chain_is_flagged_alone(p):
    import torch

    from openmcmc_b200 import kernels as K

    K.init_device(0)
    C, bad = 3000, 1234
    pr = _problem(C, p, EYE, seed=11 + p)
    pr["stats"][bad, (p - 1) * p + p - 1] = -1e6          # G[p-1][p-1] of one chain: Q not positive definite
    status = torch.zeros(C, dtype=torch.int32, device="cuda")
    beta, _ = _draw(pr, z=pr["z"], status=status)
    st = status.cpu().numpy()
    assert st[bad] != 0 and np.count_nonzero(st) == 1
    assert bool(torch.isnan(beta[bad]).all())
    ok = torch.ones(C, dtype=torch.bool, device="cuda")
    ok[bad] = False
    pr_ok = {k: (v[ok] if torch.is_tensor(v) and v.dim() > 0 and v.shape[0] == C else v) for k, v in pr.items()}
    assert _rel(beta[ok], _reference(pr_ok, pr["z"][ok])) <= 1e-9
    # solve-only mode falls back to the origin for that chain
    zero, _ = _draw(pr, solve_only=True, ridge=1e-12)
    assert float(zero[bad].abs().max()) == 0.0


@pytest.mark.parametrize("p", [64, 63, 48, 8])
def test_rss_epilogue_matches_explicit_quadratic_form(p):
    import torch

    from openmcmc_b200 import kernels as K

    K.init_device(0)
    C = 2100
    pr = _problem(C, p, EYE, seed=5 + p)
    g = torch.Generator(device="cuda").manual_seed(p)
    bhat = torch.randn(C, p, dtype=torch.float64, device="cuda", generator=g)
    c0 = torch.randn(C, p, dtype=torch.float64, device="cuda", generator=g)
    rss0 = torch.rand(C, 1, dtype=torch.float64, device="cuda", generator=g) * 100.0 + 1.0
    center = torch.cat([bhat, c0, rss0, torch.zeros(C, 1, dtype=torch.float64, device="cuda")], dim=1).contiguous()
    beta, stats = _draw(pr, z=pr["z"], center=center, rss_out=True)
    d = beta - bhat
    ref = rss0[:, 0] - 2.0 * (d * c0).sum(1) + (d.unsqueeze(1) @ pr["G"] @ d.unsqueeze(-1)).view(-1)
    got = stats[:, p * p + p]
    assert float(((got - ref).abs() / ref.abs()).max()) <= 1e-10


@pytest.mark.parametrize("p", [64, 57, 8])
def test_slice_with_chain_offset_is_bit_identical(p):
    from openmcmc_b200 import kernels as K

    K.init_device(0)
    C, lo, hi = 4096, 1500, 2700
    pr = _problem(C, p, EYE, seed=3 + p)
    full, _ = _draw(pr, rng=K.rng(seed=9, site=2))
    part, _ = _draw(pr, rng=K.rng(seed=9, chain_offset=lo, site=2), chains=slice(lo, hi))
    assert bool((full[lo:hi] == part).all())
