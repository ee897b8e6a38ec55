"""GPU parity of the left-looking warp draw (40 < p <= 64) on ill-conditioned precisions.

The kernel forms the panel below each diagonal block as a product with the inverted diagonal block and runs the
backward solve through the same inverses, instead of substituting.  Both are backward stable for the SPD diagonal
blocks of a Cholesky factorisation, but the forward error of either grows with cond(Q): this test builds Q = G + lam*I
from a skewed spectrum (eigenvalues log-spaced over cond(Q) = 1e6 ... 1e10, random eigenvectors, lam negligible) and
compares x = L^-T (L^-1 b + z) with torch's fp64 Cholesky and triangular solves, at a tolerance proportional to cond(Q).
"""

import math

import pytest

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("cond", [1e6, 1e8, 1e10])
@pytest.mark.parametrize("p", [48, 64])
def test_illconditioned_draw_matches_torch(p, cond):
    import torch

    from openmcmc_b200 import kernels as K

    K.init_device(0)
    C, dev, f64 = 300, "cuda", torch.float64
    g = torch.Generator(device=dev).manual_seed(p + round(math.log10(cond)))
    U, _ = torch.linalg.qr(torch.randn(C, p, p, dtype=f64, device=dev, generator=g))
    ev = torch.logspace(0.0, -math.log10(cond), p, dtype=f64, device=dev)
    ev = ev[torch.randperm(p, device=dev, generator=g)]
    G = (U * ev) @ U.transpose(1, 2)
    G = 0.5 * (G + G.transpose(1, 2))
    gv = torch.randn(C, p, dtype=f64, device=dev, generator=g)
    stats = torch.cat([G.reshape(C, -1), gv, torch.zeros(C, 2, dtype=f64, device=dev)], dim=1).contiguous()
    tau = torch.ones(C, dtype=f64, device=dev)
    lam = torch.full((C,), 1e-6 / cond, dtype=f64, device=dev)
    mu0 = torch.zeros(C, p, dtype=f64, device=dev)
    z = torch.randn(C, p, dtype=f64, device=dev, generator=g)
    beta = torch.empty(C, p, dtype=f64, device=dev)
    status = torch.zeros(C, dtype=torch.int32, device=dev)
    K.nn_dense_draw(C, p, stats, K.vec(tau, 1), K.MAT_EYE, K.vec(None), K.vec(lam, 1), K.vec(mu0, p), beta,
                    K.rng(seed=3, site=1), debug_z=z, status=status)
    torch.cuda.synchronize()
    assert int(status.count_nonzero()) == 0

    Q = G + lam.view(-1, 1, 1) * torch.eye(p, dtype=f64, device=dev)
    L = torch.linalg.cholesky(Q)
    w = torch.linalg.solve_triangular(L, gv.unsqueeze(-1), upper=False) + z.unsqueeze(-1)
    ref = torch.linalg.solve_triangular(L.transpose(1, 2), w, upper=True).squeeze(-1)
    kappa = torch.linalg.cond(Q)
    rel = (beta - ref).abs().amax(dim=1) / ref.abs().amax(dim=1)
    # both sides carry their own forward error, measured at up to 2e-17 cond(Q) for substitution and for this form
    assert bool((rel <= 2e-15 * kappa).all()), float((rel / kappa).max())
