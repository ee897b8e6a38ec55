"""CPU check of the lane-level model of the left-looking warp Cholesky (tools/gen/warp_chol_model.py, `run_left`):
the diagonal blocks factored with an identity tile riding along, the panel as a product with L_kk^-T, the inverted
diagonal blocks and the block mat-vec backward solve, against numpy's Cholesky and scipy's triangular solves."""

import importlib.util
import os

import numpy as np
import pytest
from scipy.linalg import solve_triangular

_PATH = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "gen", "warp_chol_model.py")


def _model():
    spec = importlib.util.spec_from_file_location("warp_chol_model", _PATH)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.parametrize("p", [48, 56, 57, 63, 64])
def test_left_model_matches_numpy(p):
    m = _model()
    rng = np.random.default_rng(p)
    A = rng.standard_normal((p, 2 * p + 3))
    Q = A @ A.T / (2 * p + 3) + 0.5 * np.eye(p)
    b, z = rng.standard_normal(p), rng.standard_normal(p)
    x, L, Linv = m.run_left(Q, b, z, (p + 7) // 8)

    Lref = np.linalg.cholesky(Q)
    assert np.max(np.abs(L - Lref)) <= 1e-13 * np.max(np.abs(Lref))
    for k in range(0, p, 8):
        blk = slice(k, min(k + 8, p))
        inv = solve_triangular(Lref[blk, blk], np.eye(blk.stop - k), lower=True)
        assert np.max(np.abs(Linv[blk, blk] - inv)) <= 1e-13 * np.max(np.abs(inv))
    # only the diagonal blocks of Linv are set
    mask = np.zeros((p, p), dtype=bool)
    for k in range(0, p, 8):
        mask[k:k + 8, k:k + 8] = True
    assert not np.any(Linv[~mask])

    ref = solve_triangular(Lref.T, solve_triangular(Lref, b, lower=True) + z, lower=False)
    assert np.max(np.abs(x - ref)) <= 1e-13 * np.max(np.abs(ref))
