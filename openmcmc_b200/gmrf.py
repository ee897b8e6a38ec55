"""Host-side mirror of `openmcmc.gmrf` for the functions on the per-sweep path (SURVEY §8 a7-a11, a21).  ref: gmrf.py

Same names and argument meaning as the reference; factorisations, solves, draws and densities run in the CUDA kernels
behind the C-ABI (`include/omc.h`); what stays in numpy is argument set-up of the one-call forms (bounds broadcasting,
`b = Q mu` of sample_truncated_normal, re-forming Q from a factor handed to a function that needs Q itself).  Inside an `MCMC` run the samplers launch these kernels directly from the sweep plan; this module is the
one-call form for code that used the reference's `gmrf` functions on their own:

    precision_irregular / precision_temporal   RW1 precision of irregular locations (one-off host setup, gmrf.py:351-411)
    cholesky / sparse_cholesky / cho_solve / solve   dense (n <= 512: blocked Cholesky with a DMMA trailing update) or
                                                bidiagonal / tridiagonal of any size (gmrf.py:414-520)
    sample_normal_canonical / sample_normal     Rue & Held Alg. 2.5 draws (gmrf.py:29-61, 167-198)
    sample_truncated_normal(_rejection) / gibbs_canonical_truncated_normal   truncated draws (gmrf.py:64-164, 201-266)
    multivariate_normal_pdf                     log-density through the Cholesky factor (gmrf.py:321-348)
    truncated_normal_rv / truncated_normal_log_pdf   scipy's log-space truncnorm on the device (gmrf.py:269-318)

Keyword extras (not in the reference): `z` / `u` inject the standard-normal / uniform variates (the reference draws them
from numpy's global generator), `seed` keys the Philox generator otherwise.  There is no CPU path: every function raises
without a CUDA device.
"""

import numpy as np
import torch
from scipy import sparse

from openmcmc_b200 import kernels as K
from openmcmc_b200.engine import classify_matrix

_calls = 0   # Philox sweep counter of the one-call draws: successive calls give fresh variates


# ---------------------------------------------------------------------------------------------- precision builders
def precision_irregular(s, is_sparse: bool = True):
    """First-order random-walk precision for irregular locations `s` (Rue & Held 2005, pp. 97-99): with gaps
    d_i = s_{i+1} - s_i the diagonal is 1/d_{i-1} + 1/d_i (one term at either end) and the off-diagonals are -1/d_i.
    Sparse CSC by default, dense otherwise; a single location gives [[1]].  ref: gmrf.py:375-411"""
    s = np.asarray(s, dtype=np.float64).reshape(-1)
    if s.size <= 1:
        return np.array(1, ndmin=2)
    inv_gap = 1.0 / (s[1:] - s[:-1])
    main = np.zeros(s.size)
    main[:-1] += inv_gap
    main[1:] += inv_gap
    if is_sparse:
        return sparse.diags([-inv_gap, main, -inv_gap], offsets=[-1, 0, 1], format="csc")
    return np.diag(main) - np.diag(inv_gap, k=-1) - np.diag(inv_gap, k=1)


def precision_temporal(time, unit_length: float = 1.0, is_sparse: bool = True):
    """`precision_irregular` on a vector of times (pandas DatetimeIndex / DatetimeArray), measured in units of
    `unit_length` seconds from the earliest one.  ref: gmrf.py:351-372"""
    seconds = np.asarray((time - time.min()).total_seconds(), dtype=np.float64) / unit_length
    return precision_irregular(seconds, is_sparse=is_sparse)


# ---------------------------------------------------------------------------------------------- helpers
def _dev():
    return torch.device("cuda", K.init_device(None))


def _t(a, dev):
    return torch.as_tensor(np.array(a, dtype=np.float64, order="C", copy=True)).to(dev)


def _dense_of(kind, main, n):
    return np.eye(n) if kind == "eye" else np.diag(main) if kind == "diag" else np.asarray(main, dtype=np.float64)


def _dense_call(A, n, b=None, z=None, want=(), factored=False, mode=0):
    """One omc_dense_factor call on a single n x n matrix (host arrays in, dict of host arrays out)."""
    dev = _dev()
    dA = _t(np.asarray(A, dtype=np.float64).reshape(1, n, n), dev)
    out = {}
    kw = {}
    if b is not None:
        kw["b"] = _t(np.asarray(b, dtype=np.float64).reshape(1, n), dev)
    if z is not None:
        kw["z"] = _t(np.asarray(z, dtype=np.float64).reshape(1, n), dev)
    for name in want:
        out[name] = torch.empty((1, n, n) if name == "L" else (1,) if name == "logdet" else (1, n), dtype=torch.float64,
                                device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    ws = K.nn_dense_workspace(1, n)
    work = torch.empty(ws, dtype=torch.float64, device=dev) if ws else None
    K.dense_factor(dA, n, status=status, factored=factored, backward_only=mode, workspace=work, **kw, **out)
    torch.cuda.synchronize()
    if int(status.item()) & 1:
        raise np.linalg.LinAlgError("Matrix is not positive definite")
    return {k: v.cpu().numpy()[0] for k, v in out.items()}


def _tridiag_call(pd, pe, n, b=None, z=None, want_logdet=False, want_factor=False, draw=True, seed=0):
    """The tridiagonal kernels on ONE system with Q = 1*P + 0*W, b = 1*h + 0: returns dict(mean, x, logdet, l, c)."""
    global _calls
    dev = _dev()
    dpd, dpe = _t(pd, dev), _t(pe if n > 1 else np.zeros(0), dev)
    zeros = torch.zeros(1, n, dtype=torch.float64, device=dev)
    h = _t(np.zeros(n) if b is None else np.asarray(b, dtype=np.float64).reshape(n), dev).reshape(1, n)
    tau0 = torch.zeros(1, dtype=torch.float64, device=dev)
    sweep = torch.full((1,), _calls, dtype=torch.int64, device=dev)
    _calls += 1
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    ws = torch.zeros(K.tridiag_workspace(1, n), dtype=torch.uint8, device=dev)
    common = dict(tau=K.vec(tau0, 1), y=K.vec(zeros, n), h=K.vec(h, n), status=status,
                  rng_=K.rng(seed=seed, sweep=sweep, site=1))
    out = {}
    mean = torch.empty(1, n, dtype=torch.float64, device=dev)
    ld = torch.zeros(1, dtype=torch.float64, device=dev)
    pl = torch.empty(1, n, dtype=torch.float64, device=dev) if want_factor else None
    pc = torch.empty(1, max(n - 1, 1), dtype=torch.float64, device=dev) if want_factor else None
    # the posterior mean is the draw with z = 0
    K.tridiag_nn_draw(K.tridiag_args(1, n, dpd, dpe, ws, **common, x=mean, debug_z=torch.zeros_like(mean),
                                     logdet=ld if want_logdet else None, probe_l=pl, probe_c=pc))
    x = None
    if draw:
        x = torch.empty_like(mean)
        dz = None if z is None else _t(np.asarray(z, dtype=np.float64).reshape(1, n), dev)
        K.tridiag_nn_draw(K.tridiag_args(1, n, dpd, dpe, ws, **common, x=x, debug_z=dz))
    torch.cuda.synchronize()
    if int(status.item()) & 1:
        raise np.linalg.LinAlgError("Matrix is not positive definite")
    out["mean"] = mean.cpu().numpy().reshape(n)
    if x is not None:
        out["x"] = x.cpu().numpy().reshape(n)
    out["logdet"] = float(ld.item())
    if want_factor:
        out["l"], out["c"] = pl.cpu().numpy().reshape(n), pc.cpu().numpy().reshape(-1)[: n - 1]
    return out


def _bidiagonal_of(L):
    """(diagonal, sub-diagonal) of a sparse lower bidiagonal factor, or None when L has another pattern."""
    L = L.tocsc(copy=True)
    L.sum_duplicates()
    L.eliminate_zeros()
    d, c = L.diagonal(0), L.diagonal(-1)
    if L.nnz != np.count_nonzero(d) + np.count_nonzero(c):
        return None
    return d, c


def _tridiag_from_factor(L):
    """Diagonals of Q = L L' for a sparse lower bidiagonal L, formed on the device (omc_bidiag_gram)."""
    bd = _bidiagonal_of(L)
    if bd is None:
        raise NotImplementedError("sparse Cholesky factors other than lower bidiagonal are not supported by the device path")
    dev = _dev()
    n = L.shape[0]
    l, c = _t(bd[0], dev), _t(bd[1], dev)
    pd = torch.empty(n, dtype=torch.float64, device=dev)
    pe = torch.empty(max(n - 1, 1), dtype=torch.float64, device=dev)
    K.bidiag_gram(l, c, n, pd, pe)
    torch.cuda.synchronize()
    return pd.cpu().numpy(), pe.cpu().numpy()[: n - 1]


def _system(Q=None, L=None):
    """Normalise (Q | L) into ("tridiag", pd, pe, n) or ("dense", matrix, factored, n)."""
    if Q is None and L is None:
        raise ValueError("either the precision Q or its Cholesky factor L is needed")
    if Q is None:
        n = L.shape[0]
        if sparse.issparse(L):
            pd, pe = _tridiag_from_factor(L)
            return ("tridiag", pd, pe, n)
        return ("dense", np.asarray(L, dtype=np.float64), True, n)
    kind, main, off = classify_matrix(Q)
    n = Q.shape[0]
    if kind == "tridiag" or (kind in ("eye", "diag") and n > 512):
        return ("tridiag", np.ones(n) if kind == "eye" else main, off if kind == "tridiag" else np.zeros(max(n - 1, 0)), n)
    if n > 512:
        raise NotImplementedError(f"dense {n} x {n} precision: the device path factorises dense matrices up to 512")
    return ("dense", _dense_of(kind, main, n), False, n)


# ---------------------------------------------------------------------------------------------- factorisation / solves
def cholesky(Q, lower: bool = True):
    """Cholesky factor in the format of the input: dense `Q` -> dense L (blocked Cholesky with a DMMA trailing update,
    omc_dense_factor), sparse tridiagonal / diagonal `Q` -> sparse bidiagonal L (the tridiagonal kernels' factor
    probes).  `lower=False` gives L'.  ref: gmrf.py:465-486"""
    if sparse.issparse(Q):
        L = sparse_cholesky(Q)
    else:
        Qd = np.asarray(Q, dtype=np.float64)
        L = _dense_call(Qd, Qd.shape[0], want=("L",))["L"]
    return L if lower else L.T


def sparse_cholesky(Q):
    """Natural-order Cholesky of a sparse SPD matrix as a sparse CSC factor (the reference: SuperLU without pivoting,
    L diag(U)^1/2).  Tridiagonal and diagonal patterns run on the tridiagonal kernels; any other pattern up to
    512 x 512 is factorised densely on the device.  ref: gmrf.py:489-520"""
    if Q.shape[0] != Q.shape[1]:
        raise ValueError("Matrix is not square")
    sysm = _system(Q=Q)
    n = sysm[-1]
    if sysm[0] == "tridiag":
        r = _tridiag_call(sysm[1], sysm[2], n, want_factor=True, draw=False)
        return sparse.diags([r["c"], r["l"]], offsets=[-1, 0], format="csc") if n > 1 else sparse.csc_matrix(r["l"].reshape(1, 1))
    return sparse.csc_matrix(_dense_call(sysm[1], n, want=("L",))["L"])


def cho_solve(c_and_lower: tuple, b):
    """Solve A x = b given the Cholesky factor of A (`(c, lower)` as scipy's cho_solve).  ref: gmrf.py:437-462"""
    c, lower = c_and_lower
    Lf = c if lower else c.T
    bs = b.toarray() if sparse.issparse(b) else np.asarray(b, dtype=np.float64)
    cols = bs.reshape(bs.shape[0], -1)
    sysm = _system(L=Lf)
    n = sysm[-1]
    out = np.empty_like(cols, dtype=np.float64)
    for j in range(cols.shape[1]):
        if sysm[0] == "tridiag":
            out[:, j] = _tridiag_call(sysm[1], sysm[2], n, b=cols[:, j], draw=False)["mean"]
        else:
            out[:, j] = _dense_call(sysm[1], n, b=cols[:, j], want=("mean",), factored=True)["mean"]
    return out.reshape(bs.shape)


def solve(a, b):
    """Solution of a x = b for the systems the hot path meets: `a` triangular (the `solve(L.T, z)` of sample_normal,
    gmrf.py:61) or symmetric positive definite; dense up to 512, sparse bidiagonal / tridiagonal of any size.  A
    general non-symmetric `a` (LU in the reference) is outside the device path.  ref: gmrf.py:414-434"""
    bs = b.toarray() if sparse.issparse(b) else np.asarray(b, dtype=np.float64)
    cols = bs.reshape(bs.shape[0], -1)
    n = a.shape[0]
    out = np.empty_like(cols, dtype=np.float64)
    if sparse.issparse(a):
        if sparse.triu(a, 1).nnz == 0 or sparse.tril(a, -1).nnz == 0:
            raise NotImplementedError("gmrf.solve with a sparse triangular matrix: hand the factor to cho_solve / "
                                      "sample_normal(L=...) instead (they run the bidiagonal substitutions on the device)")
        sysm = _system(Q=a)
        for j in range(cols.shape[1]):
            out[:, j] = (_tridiag_call(sysm[1], sysm[2], n, b=cols[:, j], draw=False)["mean"] if sysm[0] == "tridiag"
                         else _dense_call(sysm[1], n, b=cols[:, j], want=("mean",))["mean"])
        return out.reshape(bs.shape)
    ad = np.asarray(a, dtype=np.float64)
    if not np.any(np.tril(ad, -1)):           # upper triangular: a = L'
        mode, Lf, fact = 1, ad.T, True
    elif not np.any(np.triu(ad, 1)):          # lower triangular: a = L
        mode, Lf, fact = 2, ad, True
    elif np.array_equal(ad, ad.T):
        mode, Lf, fact = 0, ad, False
    else:
        raise NotImplementedError("gmrf.solve on the device handles triangular and symmetric positive definite systems")
    for j in range(cols.shape[1]):
        out[:, j] = _dense_call(Lf, n, b=cols[:, j], want=("mean",), factored=fact, mode=mode)["mean"]
    return out.reshape(bs.shape)


def _factor_and_solve(Q, b, z, seed, want_logdet=False, L=None):
    """One chain: mu = Q^-1 b, x = mu + L^-T z (z = None: Philox normals) on the device.  Returns (x, mu, logdet)."""
    global _calls
    sysm = _system(Q=Q, L=L)
    n = sysm[-1]
    b = np.zeros(n) if b is None else np.asarray(b, dtype=np.float64).reshape(-1)
    if b.size != n:
        raise ValueError(f"b has {b.size} entries for a {n} x {n} precision")
    if sysm[0] == "tridiag":
        r = _tridiag_call(sysm[1], sysm[2], n, b=b, z=z, want_logdet=want_logdet, seed=seed,
                          draw=(z is not None or not want_logdet))
        x = r.get("x", r["mean"])
        return x.reshape(n, 1), r["mean"].reshape(n, 1), r["logdet"]
    if z is None:            # free-running normals: the sweep kernel draws them (Philox, keyed by the call counter)
        dev = _dev()
        rec = torch.zeros(1, n * n + n + 2, dtype=torch.float64, device=dev)
        A = sysm[1] @ sysm[1].T if sysm[2] else sysm[1]          # (a given dense factor: Q re-formed for this path only)
        rec[0, : n * n] = _t(np.asarray(A).reshape(-1), dev)
        rec[0, n * n: n * n + n] = _t(b, dev)
        one, zero = torch.ones(1, dtype=torch.float64, device=dev), torch.zeros(1, dtype=torch.float64, device=dev)
        x = torch.empty(1, n, dtype=torch.float64, device=dev)
        mu = torch.empty(1, n, dtype=torch.float64, device=dev)
        Lp = torch.empty(1, n, n, dtype=torch.float64, device=dev)
        sweep = torch.full((1,), _calls, dtype=torch.int64, device=dev)
        _calls += 1
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        ws = K.nn_dense_workspace(1, n)
        work = torch.empty(ws, dtype=torch.float64, device=dev) if ws else None
        K.nn_dense_draw(1, n, rec, K.vec(one, 1), K.MAT_EYE, K.vec(None), K.vec(zero, 1), K.vec(None), x,
                        K.rng(seed=seed, sweep=sweep, site=1), probe_mu=mu, probe_L=Lp, status=status, workspace=work)
        torch.cuda.synchronize()
        if int(status.item()) & 1:
            raise np.linalg.LinAlgError("Matrix is not positive definite")
        ld = 0.0
        if want_logdet:
            ld = _dense_call(A, n, want=("logdet",))["logdet"]
        return x.cpu().numpy().reshape(n, 1), mu.cpu().numpy().reshape(n, 1), float(np.ravel(ld)[0]) if want_logdet else 0.0
    want = ("mean", "x") + (("logdet",) if want_logdet else ())
    r = _dense_call(sysm[1], n, b=b, z=z, want=want, factored=sysm[2])
    return r["x"].reshape(n, 1), r["mean"].reshape(n, 1), float(np.ravel(r["logdet"])[0]) if want_logdet else 0.0


# ---------------------------------------------------------------------------------------------- draws
def sample_normal_canonical(b, Q=None, L=None, z=None, seed: int = 0):
    """x ~ N(Q^-1 b, Q^-1) by Rue & Held Alg. 2.5: L = chol(Q), L w = b, L' mu = w, L' v = z, x = mu + v.
    `Q` dense (up to 512) or sparse diagonal / tridiagonal of any size; a precomputed factor `L` (dense, or sparse
    bidiagonal) is used as it is.  Returns a p x 1 array.  ref: gmrf.py:167-198"""
    x, _, _ = _factor_and_solve(Q, b, z, seed, L=L if Q is None else None)
    return x.reshape(np.shape(b)) if np.ndim(b) == 2 else x


def sample_normal(mu, Q=None, L=None, n: int = 1, z=None, seed: int = 0):
    """x ~ N(mu, Q^-1): mu + L^-T z, one column per draw.  Returns p x n.  ref: gmrf.py:29-61"""
    mu = np.asarray(mu, dtype=np.float64).reshape(-1, 1)
    cols = []
    for j in range(n):
        zj = None if z is None else np.asarray(z, dtype=np.float64).reshape(mu.size, -1)[:, j]
        x, _, _ = _factor_and_solve(Q, None, zj, seed, L=L if Q is None else None)
        cols.append(x + mu)
    return np.concatenate(cols, axis=1)


def gibbs_canonical_truncated_normal(b, Q, x, lower=-np.inf, upper=np.inf, u=None, seed: int = 0):
    """One coordinate-wise Gibbs scan of N_c(Q^-1 b, Q^-1) truncated to [lower, upper] from the current `x`
    (Rue & Held 2005, Lemma 2.1): x_i ~ N(v_i (b_i - Q_i. x + Q_ii x_i), v_i = 1 / Q_ii) truncated, one truncnorm
    inverse-CDF draw per coordinate (`u`: the uniforms behind them).  Unbounded: a plain canonical draw.  The scan is
    the truncated-prior mode of omc_nn_dense_draw: Q in shared memory up to p = 64, the rows of Q streamed through
    shared memory by one warp above that, up to p = 512.  ref: gmrf.py:201-266"""
    def unbounded(v, inf):
        return v is None or (np.ndim(v) == 0 and v == inf)

    if unbounded(lower, -np.inf) and unbounded(upper, np.inf):
        return sample_normal_canonical(b, Q, seed=seed)
    global _calls
    dev = _dev()
    Qd = Q.toarray() if sparse.issparse(Q) else np.asarray(Q, dtype=np.float64)
    p = Qd.shape[0]
    if p > 512:
        raise NotImplementedError(f"gibbs_canonical_truncated_normal on the device supports p <= 512 (p = {p})")
    rec = torch.zeros(1, p * p + p + 2, dtype=torch.float64, device=dev)
    rec[0, : p * p] = _t(Qd.reshape(-1), dev)
    rec[0, p * p: p * p + p] = _t(np.asarray(b, dtype=np.float64).reshape(-1), dev)
    one, zero = torch.ones(1, dtype=torch.float64, device=dev), torch.zeros(1, dtype=torch.float64, device=dev)
    xd = _t(np.asarray(x, dtype=np.float64).reshape(1, p), dev)
    lo = _t(np.broadcast_to(np.asarray(-np.inf if lower is None else lower, dtype=np.float64).reshape(-1, 1), (p, 1)).reshape(-1), dev)
    hi = _t(np.broadcast_to(np.asarray(np.inf if upper is None else upper, dtype=np.float64).reshape(-1, 1), (p, 1)).reshape(-1), dev)
    du = None if u is None else _t(np.asarray(u, dtype=np.float64).reshape(1, p), dev)
    sweep = torch.full((1,), _calls, dtype=torch.int64, device=dev)
    _calls += 1
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    K.nn_dense_draw(1, p, rec, K.vec(one, 1), K.MAT_EYE, K.vec(None), K.vec(zero, 1), K.vec(None), xd,
                    K.rng(seed=seed, sweep=sweep, site=2), status=status, trunc=(K.vec(lo), p, K.vec(hi), p), debug_u=du)
    torch.cuda.synchronize()
    return xd.cpu().numpy().reshape(p, 1)


def sample_truncated_normal_rejection(mu, Q=None, L=None, lower=None, upper=None, n: int = 1, seed: int = 0):
    """Rejection sampling from N(mu, Q^-1) truncated to [lower, upper]: unconstrained draws (device), columns outside
    the box redrawn until none is left.  ref: gmrf.py:113-164"""
    lower = -np.inf if lower is None else lower
    upper = np.inf if upper is None else upper
    if np.any(np.asarray(lower) >= np.asarray(upper)):
        raise ValueError("Error lower bound must be strictly less than upper bound")
    samples = sample_normal(mu, Q=Q, L=L, n=n, seed=seed)
    bad = np.any((samples < lower) | (samples > upper), axis=0)
    while bad.any():
        samples[:, bad] = sample_normal(mu, Q=Q, L=L, n=int(bad.sum()), seed=seed)
        bad = np.any((samples < lower) | (samples > upper), axis=0)
    return samples


def sample_truncated_normal(mu, Q=None, L=None, lower=None, upper=None, n: int = 1, method="Gibbs", seed: int = 0):
    """Truncated multivariate normal draws: `Gibbs` (a rejection draw to start, then 10 coordinate-wise scans between
    kept draws) or `Rejection`.  ref: gmrf.py:64-110"""
    if method == "Gibbs":
        mu = np.asarray(mu, dtype=np.float64).reshape(-1, 1)
        if Q is None:
            Ld = L.toarray() if sparse.issparse(L) else np.asarray(L, dtype=np.float64)
            Q = Ld @ Ld.T            # the scan needs Q itself (one-off set-up, as the reference's `Q @ mu`)
        Qd = Q.toarray() if sparse.issparse(Q) else np.asarray(Q, dtype=np.float64)
        b = Qd @ mu
        d = mu.shape[0]
        Z = np.empty((d, n))
        Z[:, 0] = sample_truncated_normal_rejection(mu, Q=Qd, lower=lower, upper=upper, n=1, seed=seed).ravel()
        for i in range(n - 1):
            x = Z[:, i].reshape(d, 1)
            for _ in range(10):
                x = gibbs_canonical_truncated_normal(b, Qd, x, lower=lower, upper=upper, seed=seed)
            Z[:, i + 1] = x.ravel()
        return Z
    if method == "Rejection":
        return sample_truncated_normal_rejection(mu, Q=Q, L=L, lower=lower, upper=upper, n=n, seed=seed)
    raise TypeError("method should be either Gibbs or Rejection")


def multivariate_normal_pdf(x, mu, Q, by_observation: bool = False):
    """Log-density of N(mu, Q^-1) at the columns of x (dim x n): 1/2 (log|Q| - dim log 2 pi - |L'(x - mu)|^2); summed
    over the observations unless `by_observation`.  log|Q| comes from the device factorisation, the quadratic forms
    (x - mu)' Q (x - mu) = |L'(x - mu)|^2 from `omc_quadform` / `omc_tridiag_matvec`.  ref: gmrf.py:321-348"""
    x = np.asarray(x, dtype=np.float64)
    x = x.reshape(-1, 1) if x.ndim == 1 else x
    mu = np.asarray(mu, dtype=np.float64).reshape(-1, 1)
    dim, n_obs = x.shape
    _, _, logdet = _factor_and_solve(Q, None, np.zeros(dim), 0, want_logdet=True)
    # quadratic forms (x_r - mu)' Q (x_r - mu) on the device, one observation per "chain" of the kernel
    dev = _dev()
    kind, main, off = classify_matrix(Q)
    xd, mud = _t(x.T, dev), _t(mu.reshape(-1), dev)                 # [n_obs, dim], [dim]
    quad = torch.empty(n_obs, dtype=torch.float64, device=dev)
    if kind == "tridiag":
        r = (xd - mud).contiguous()
        Qr = torch.empty_like(r)
        K.tridiag_matvec(_t(main, dev), _t(off, dev), K.vec(r, dim), n_obs, dim, Qr)
        quad = (r * Qr).sum(dim=1)
    else:
        cnt = torch.empty(n_obs, dtype=torch.float64, device=dev)
        if kind == "eye":
            K.quadform(n_obs, dim, K.vec(xd, dim), K.vec(mud, 0), K.MAT_EYE, K.vec(None), quad, cnt)
        elif kind == "diag":
            K.quadform(n_obs, dim, K.vec(xd, dim), K.vec(mud, 0), K.MAT_DIAG, K.vec(_t(main, dev), 0), quad, cnt)
        else:
            K.quadform(n_obs, dim, K.vec(xd, dim), K.vec(mud, 0), K.MAT_DENSE, K.vec(_t(np.asarray(main), dev), 0), quad, cnt)
    torch.cuda.synchronize()
    log_p = 0.5 * (logdet - dim * np.log(2.0 * np.pi) - quad.cpu().numpy().reshape(-1))
    return log_p if by_observation else np.sum(log_p)


# ---------------------------------------------------------------------------------------------- truncated normal
def _bcast(v, shape, default):
    return np.broadcast_to(np.asarray(default if v is None else v, dtype=np.float64), shape).reshape(-1)


def truncated_normal_rv(mean, scale, lower, upper, size=1, u=None, seed: int = 0):
    """Truncated-normal draws on [lower, upper] by the log-space inverse CDF scipy's `truncnorm.rvs` uses, from
    uniforms `u` (Philox when not given).  None bounds are infinite.  ref: gmrf.py:269-292"""
    if np.ndim(size) > 0:
        shape = tuple(int(v) for v in size)
    elif int(size) != 1:
        shape = (int(size),)
    else:
        shape = np.broadcast(np.asarray(mean, dtype=np.float64), np.asarray(scale, dtype=np.float64)).shape or (1,)
    n = int(np.prod(shape))
    dev = _dev()
    if u is None:
        gen = torch.Generator(device=dev)
        gen.manual_seed(int(seed) + 7919 * (_calls_bump()))
        ud = torch.rand(n, dtype=torch.float64, device=dev, generator=gen)
    else:
        ud = _t(_bcast(u, shape, 0.5), dev)
    out = torch.empty(n, dtype=torch.float64, device=dev)
    K.truncnorm_rv(_t(_bcast(mean, shape, 0.0), dev), _t(_bcast(scale, shape, 1.0), dev),
                   _t(_bcast(lower, shape, -np.inf), dev), _t(_bcast(upper, shape, np.inf), dev), ud, out)
    return out.cpu().numpy().reshape(shape)


def truncated_normal_log_pdf(x, mean, scale, lower, upper):
    """log-pdf of the truncated normal (scipy's `truncnorm.logpdf`: -inf outside the bounds).  ref: gmrf.py:295-318"""
    x = np.asarray(x, dtype=np.float64)
    shape = np.broadcast(x, np.asarray(mean, dtype=np.float64), np.asarray(scale, dtype=np.float64)).shape
    dev = _dev()
    out = torch.empty(int(np.prod(shape)), dtype=torch.float64, device=dev)
    K.truncnorm_logpdf(_t(_bcast(x, shape, 0.0), dev), _t(_bcast(mean, shape, 0.0), dev), _t(_bcast(scale, shape, 1.0), dev),
                       _t(_bcast(lower, shape, -np.inf), dev), _t(_bcast(upper, shape, np.inf), dev), out)
    return out.cpu().numpy().reshape(shape)


def _calls_bump():
    global _calls
    _calls += 1
    return _calls
