"""The left-looking warp draw (40 < p <= 64) with its operands in accumulator order.

The kernel takes each tile product's k index in the order k = 2kq + s of m8n8k4 step s, so every operand fragment is
a lane's own accumulator element and the factor's tiles are stored and read back as one 16-byte access per lane, and
its rss epilogue takes d from the backward solve's registers.  Checked here, at block counts 6, 7 and 8 with full and
ragged last blocks:

* injected-z draws against torch's fp64 Cholesky and triangular solves on precisions of condition 1e2 ... 1e10, at a
  tolerance proportional to cond(Q);
* rss = rss0 - 2 d'c0 + d'G d against a long-double evaluation at the returned beta, within 64 eps of its terms;
* bit equality of two launches, and of a slice of chains launched alone with the RNG's chain offset.
"""

import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PS = [41, 48, 57, 63, 64]


def _problem(C, p, cond, seed):
    """Q = G + lam I with G's eigenvalues log-spaced over [1 / cond, 1] (random eigenvectors, lam negligible)."""
    import torch

    dev, f64 = "cuda", torch.float64
    g = torch.Generator(device=dev).manual_seed(seed)
    U, _ = torch.linalg.qr(torch.randn(C, p, p, dtype=f64, device=dev, generator=g))
    ev = torch.logspace(0.0, -math.log10(cond), p, dtype=f64, device=dev)
    ev = ev[torch.randperm(p, device=dev, generator=g)]
    G = (U * ev) @ U.transpose(1, 2)
    G = 0.5 * (G + G.transpose(1, 2))
    gv = torch.randn(C, p, dtype=f64, device=dev, generator=g)
    stats = torch.cat([G.reshape(C, -1), gv, torch.zeros(C, 2, dtype=f64, device=dev)], dim=1).contiguous()
    lam = torch.full((C,), 1e-6 / cond, dtype=f64, device=dev)
    z = torch.randn(C, p, dtype=f64, device=dev, generator=g)
    bhat = torch.randn(C, p, dtype=f64, device=dev, generator=g)
    c0 = torch.randn(C, p, dtype=f64, device=dev, generator=g)
    rss0 = torch.rand(C, 1, dtype=f64, device=dev, generator=g) * 100.0 + 1.0
    center = torch.cat([bhat, c0, rss0, torch.zeros(C, 1, dtype=f64, device=dev)], dim=1).contiguous()
    return dict(C=C, p=p, G=G, gv=gv, stats=stats, lam=lam, z=z, center=center)


def _draw(pr, z=None, rng=None, chains=None, rss=False):
    import torch

    from openmcmc_b200 import kernels as K

    p = pr["p"]
    sl = slice(0, pr["C"]) if chains is None else chains
    n = sl.stop - sl.start
    stats = pr["stats"][sl].clone()
    beta = torch.empty(n, p, dtype=torch.float64, device="cuda")
    status = torch.zeros(n, dtype=torch.int32, device="cuda")
    mu0 = torch.zeros(p, dtype=torch.float64, device="cuda")
    K.nn_dense_draw(n, p, stats, K.vec(torch.ones(n, dtype=torch.float64, device="cuda"), 1), K.MAT_EYE, K.vec(None),
                    K.vec(pr["lam"][sl].contiguous(), 1), K.vec(mu0, 0), beta,
                    rng if rng is not None else K.rng(seed=5, site=1), debug_z=None if z is None else z[sl].contiguous(),
                    status=status, center=pr["center"][sl].contiguous() if rss else None,
                    rss_out=stats.data_ptr() + 8 * (p * p + p) if rss else None)
    torch.cuda.synchronize()
    assert int(status.count_nonzero()) == 0
    return beta, stats[:, p * p + p]


@pytest.mark.parametrize("cond", [1e2, 1e6, 1e10])
@pytest.mark.parametrize("p", PS)
def test_injected_z_matches_torch(p, cond):
    import torch

    from openmcmc_b200 import kernels as K

    K.init_device(0)
    pr = _problem(300, p, cond, seed=31 * p + round(math.log10(cond)))
    beta, _ = _draw(pr, z=pr["z"])
    Q = pr["G"] + pr["lam"].view(-1, 1, 1) * torch.eye(p, dtype=torch.float64, device="cuda")
    L = torch.linalg.cholesky(Q)
    w = torch.linalg.solve_triangular(L, pr["gv"].unsqueeze(-1), upper=False) + pr["z"].unsqueeze(-1)
    ref = torch.linalg.solve_triangular(L.transpose(1, 2), w, upper=True).squeeze(-1)
    kappa = torch.linalg.cond(Q)
    rel = (beta - ref).abs().amax(dim=1) / ref.abs().amax(dim=1)
    assert bool((rel <= 1e-15 * kappa).all()), float((rel / kappa).max())


@pytest.mark.parametrize("p", PS)
def test_rss_matches_long_double(p):
    from openmcmc_b200 import kernels as K

    K.init_device(0)
    C = 200
    pr = _problem(C, p, 1e4, seed=7 + p)
    beta, rss = _draw(pr, z=pr["z"], rss=True)
    ld = np.longdouble
    b = beta.cpu().numpy().astype(ld)
    cen = pr["center"].cpu().numpy().astype(ld)
    G = pr["G"].cpu().numpy().astype(ld)
    d = b - cen[:, :p]
    c0, rss0 = cen[:, p:2 * p], cen[:, 2 * p]
    lin = np.einsum("ci,ci->c", d, c0)
    quad = np.einsum("ci,cij,cj->c", d, G, d)
    ref = rss0 - 2 * lin + quad
    terms = np.abs(rss0) + 2 * np.einsum("ci,ci->c", np.abs(d), np.abs(c0)) + \
        np.einsum("ci,cij,cj->c", np.abs(d), np.abs(G), np.abs(d))
    err = np.abs(rss.cpu().numpy().astype(ld) - ref)
    eps = np.finfo(np.float64).eps
    assert bool(np.all(err <= 64 * eps * terms)), float(np.max(err / terms))


@pytest.mark.parametrize("p", PS)
def test_repeat_and_chain_offset_shard_are_bit_identical(p):
    from openmcmc_b200 import kernels as K

    K.init_device(0)
    C, lo, hi = 4096, 1500, 2700
    pr = _problem(C, p, 1e3, seed=13 + p)
    b1, r1 = _draw(pr, rng=K.rng(seed=9, site=2), rss=True)
    b2, r2 = _draw(pr, rng=K.rng(seed=9, site=2), rss=True)
    assert bool((b1 == b2).all()) and bool((r1 == r2).all())
    bs, rs = _draw(pr, rng=K.rng(seed=9, chain_offset=lo, site=2), chains=slice(lo, hi), rss=True)
    assert bool((b1[lo:hi] == bs).all()) and bool((r1[lo:hi] == rs).all())
