"""Sweep-plan compiler and resident device state.

The reference runs `for sampler in samplers: state = sampler.sample(state)` over a dict of numpy arrays
(mcmc.py:97-111).  Here the same (model, samplers, state) triple is compiled ONCE into a list of CUDA kernel launches
over buffers resident in HBM, batched over `n_chains` independent chains; the launch list of one sweep is captured in a
CUDA graph and replayed (kernels.Graph / omc_run_schedule).

Host logic only: shapes, pattern matching of the declarative model onto kernels, and a small dataflow pass that
decides which derived quantities (sufficient statistics, quadratic forms) are still valid at each point of the sweep so
that e.g. the Gibbs regression needs exactly ONE pass over X per sweep.  No arithmetic on chain state happens here.
"""

from dataclasses import dataclass, field

import numpy as np
import torch
from scipy import sparse

from openmcmc_b200 import kernels as K
from openmcmc_b200.parameter import Identity, LinearCombination, ScaledMatrix

F64 = torch.float64

# Data-only parts of a derived record (G = X'WX, g = X'Wy of the regression record) are kept across sweeps and only the
# state-dependent part (the residual sum of squares) is refreshed.  False re-runs the full fused pass (DMMA SYRK
# included) every sweep, the way the reference recomputes A'QA in every NormalNormal.sample (sampler.py:180-186);
# bench.py times that form next to the shipped one.
CACHE_DATA_ONLY = True
# With G | g cached, the residual sum of squares of the CURRENT beta needs no pass over X either: the prologue fixes a
# centre beta_hat (the least-squares point), streams X once more for c0 = X'W(y - X beta_hat) and rss0, and the draw
# kernel's epilogue evaluates rss(beta) = rss0 - 2 d'c0 + d'G d, d = beta - beta_hat (omc.h: omc_nn_dense_t.center).
# False keeps the explicit residual pass (omc_reg_rss) in every sweep; tests compare the two forms.
RECENTER = True
# Consecutive per-chain O(1) / O(p) operations of a sweep or of the store epilogue (Gamma draws, small quadratic forms,
# log-density terms, sample copies) are issued as ONE launch (omc_fused_small).  False keeps one kernel per operation.
FUSE_SMALL = True


# ============================================================================================== device state
@dataclass
class DevArray:
    """One state entry on the device.

    data : float64 tensor, [C, rows, cols] when per_chain else [rows, cols]
    kind : 'dense' | 'eye' | 'diag' | 'tridiag'   (structure of a square matrix; 'dense' for everything else)
           eye -> data None ; diag -> data [.., n] ; tridiag -> data [.., n] main diagonal and off [.., n-1]
    """

    data: torch.Tensor
    per_chain: bool
    rows: int
    cols: int
    kind: str = "dense"
    off: torch.Tensor = None
    npos: int = None          # structured matrices: number of positive diagonal entries (sampler.py:283), host count
    is_matrix: bool = False   # classified by put(as_matrix=True): structure is final, never re-uploaded

    @property
    def size(self):
        return self.rows * self.cols

    def vec(self, elems=None):
        if self.data is None:
            return K.vec(None)
        per = self.data[0].numel() if self.per_chain else None
        return K.vec(self.data, per)

    def off_vec(self):
        per = self.off[0].numel() if self.per_chain else None
        return K.vec(self.off, per)


_classify_cache = {}


def classify_matrix(m):
    """Structure of a (host) square matrix: returns (kind, main, off).  Host-side inspection of constant data; the
    result for a sparse matrix object is remembered while that object lives (a 1e6-point precision costs ~10 ms per
    inspection and the plan compiler asks several times)."""
    if sparse.issparse(m):
        import weakref

        sig = (m.nnz, m.shape, float(m.data.sum()) if m.nnz else 0.0)     # values changed in place => inspected again
        hit = _classify_cache.get(id(m))
        if hit is not None and hit[0]() is m and hit[1] == sig:
            return hit[2]
        out = _classify_matrix(m)
        try:
            _classify_cache[id(m)] = (weakref.ref(m, lambda _r, k=id(m): _classify_cache.pop(k, None)), sig, out)
        except TypeError:
            pass
        return out
    return _classify_matrix(m)


def _classify_matrix(m):
    if sparse.issparse(m):
        m = m.tocsc(copy=True)        # canonical form: duplicates summed, explicit zeros dropped
        m.sum_duplicates()
        m.eliminate_zeros()
        n = m.shape[0]
        d = m.diagonal(0)
        if m.nnz == np.count_nonzero(d):
            return ("eye", None, None) if np.all(d == 1.0) else ("diag", d, None)
        e_lo, e_up = m.diagonal(-1), m.diagonal(1)
        if m.nnz == np.count_nonzero(d) + np.count_nonzero(e_lo) + np.count_nonzero(e_up):
            if not np.array_equal(e_lo, e_up):
                raise NotImplementedError("non-symmetric tridiagonal precision matrix")
            return "tridiag", d, e_lo
        if n <= 512:
            return "dense", np.asarray(m.todense(), dtype=np.float64), None
        raise NotImplementedError(f"sparse {n}x{n} precision with bandwidth > 1 is not supported by the device path")
    m = np.asarray(m, dtype=np.float64)
    n = m.shape[0]
    if m.ndim == 2 and m.shape[0] == m.shape[1]:
        offd = m - np.diag(np.diag(m))
        if not np.any(offd):
            d = np.diag(m).copy()
            return ("eye", None, None) if np.all(d == 1.0) else ("diag", d, None)
        if n > 2 and not np.any(np.triu(m, 2)) and not np.any(np.tril(m, -2)) and n > 64:
            return "tridiag", np.diag(m).copy(), np.diag(m, -1).copy()
    return "dense", m, None


class DeviceState:
    """Chain-batched MCMC state resident in HBM (replaces the reference's dict of numpy arrays, mcmc.py:63-76).

    Entries are uploaded lazily from the bound host dict the first time a plan fragment asks for them.
    """

    def __init__(self, n_chains: int, device: int, host_state: dict = None, per_chain_names=()):
        self.n_chains = n_chains
        self.device = torch.device("cuda", device)
        self.arrays = {}
        self.host_state = host_state if host_state is not None else {}
        self.per_chain_names = set(per_chain_names)
        self.h2d_bytes = 0
        self._retired = []   # replaced entries stay alive: kernels hold raw device pointers (omc_vec_t) into them

    def _t(self, a):
        a = np.ascontiguousarray(a, dtype=np.float64)
        if not a.flags.writeable:
            a = a.copy()
        self.h2d_bytes += a.nbytes
        return K.upload(a, self.device)

    def put(self, name, value, per_chain=None, as_matrix=False):
        """Upload one entry.  2-D host arrays are shared by all chains unless per_chain=True (then replicated);
        3-D arrays [C, rows, cols] are per-chain.  torch tensors are moved/bound as they are."""
        C = self.n_chains
        if name in self.arrays:
            self._retired.append(self.arrays[name])
        if per_chain is None:
            per_chain = name in self.per_chain_names
        if isinstance(value, torch.Tensor):
            if not value.is_cuda:
                self.h2d_bytes += value.numel() * value.element_size()
            t = value.to(self.device, F64, non_blocking=True)
            if per_chain and t.data_ptr() == value.data_ptr():
                t = t.clone()   # sampled entries are written by the kernels: never alias the caller's tensor
            if t.dim() == 3:
                if t.shape[0] != C:
                    raise ValueError(f"state['{name}'] has leading dimension {t.shape[0]} but n_chains={C}")
                arr = DevArray(t.contiguous(), True, t.shape[1], t.shape[2])
            else:
                t = t.reshape(t.shape[0], -1) if t.dim() == 2 else t.reshape(-1, 1)
                if t.shape[0] == 1 and t.shape[1] > 1:
                    t = t.t()
                arr = DevArray(t.contiguous(), False, t.shape[0], t.shape[1])
                if per_chain:
                    arr = DevArray(t.unsqueeze(0).repeat(C, 1, 1).contiguous(), True, t.shape[0], t.shape[1])
            self.arrays[name] = arr
            return arr
        if as_matrix or sparse.issparse(value):
            kind, main, off = classify_matrix(value)
            n = value.shape[0]
            npos = n if kind == "eye" else int(np.sum((np.diag(main) if kind == "dense" else main) > 0))
            if kind == "eye":
                arr = DevArray(None, False, n, n, "eye")
            elif kind == "diag":
                arr = DevArray(self._t(main), False, n, n, "diag")
            elif kind == "tridiag":
                arr = DevArray(self._t(main), False, n, n, "tridiag", self._t(off))
            else:
                arr = DevArray(self._t(main), False, n, n, "dense")
            arr.is_matrix = True
            arr.npos = npos
            self.arrays[name] = arr
            return arr
        a = np.asarray(value, dtype=np.float64)
        if a.ndim == 3:
            if a.shape[0] != C:
                raise ValueError(f"state['{name}'] has leading dimension {a.shape[0]} but n_chains={C}")
            arr = DevArray(self._t(a), True, a.shape[1], a.shape[2])
        else:
            # reference coercion (mcmc.py:65-76): scalars / 1-D -> column vectors, (1,k) lists -> (k,1)
            if a.ndim < 2:
                a = np.atleast_2d(a).T
            elif a.shape[0] == 1 and a.shape[1] > 1 and not isinstance(value, np.ndarray):
                a = a.T
            if per_chain:
                arr = DevArray(self._t(np.broadcast_to(a, (C,) + a.shape)), True, a.shape[0], a.shape[1])
            else:
                arr = DevArray(self._t(a), False, a.shape[0], a.shape[1])
        self.arrays[name] = arr
        return arr

    def __getitem__(self, name):
        if name not in self.arrays:
            if name not in self.host_state:
                raise KeyError(f"state entry '{name}' is required by the model but missing from the state")
            self.put(name, self.host_state[name])
        return self.arrays[name]

    def __contains__(self, name):
        return name in self.arrays or name in self.host_state

    def get_host(self, name):
        """Download: per-chain entries come back as [C, rows, cols] (squeezed to [rows, cols] when C == 1)."""
        a = self.arrays[name]
        if a.data is None:
            return sparse.identity(a.rows, format="csc")
        h = K.download(a.data)
        if a.per_chain and self.n_chains == 1:
            h = h[0]
        return h


# ============================================================================================== plan
class PlanError(NotImplementedError):
    """The (model, sampler) combination is outside what the device path implements; raised at compile time."""


@dataclass
class Quantity:
    """A derived per-chain quantity (e.g. sufficient statistics) with the state entries it depends on."""

    name: str
    deps: frozenset
    compute: callable  # emits the kernels that refresh it (may refresh sibling quantities as well)
    siblings: tuple = ()


@dataclass
class Plan:
    """Launch list of one sweep plus the store epilogue, built for a fixed (model, samplers, state layout)."""

    state: DeviceState
    seed: int = 0
    chain_offset: int = 0
    quantities: dict = field(default_factory=dict)
    valid: dict = field(default_factory=dict)
    ops: list = field(default_factory=list)          # current emission target
    n_sites: int = 0
    sweep_counter: torch.Tensor = None
    iter_counter: torch.Tensor = None
    status: torch.Tensor = None
    debug: dict = field(default_factory=dict)         # site name -> injected draw tensors
    probes: dict = field(default_factory=dict)        # name -> tensor with intermediates (parity tests)
    keep: list = field(default_factory=list)          # tensors that must outlive the captured graph
    recenter: bool = True                             # False for one-call plans: a centre would cost 3 passes over X

    def __post_init__(self):
        dev = self.state.device
        self.sweep_counter = torch.zeros(1, dtype=torch.int64, device=dev)
        self.iter_counter = torch.zeros(1, dtype=torch.int64, device=dev)
        self.status = torch.zeros(self.state.n_chains, dtype=torch.int32, device=dev)

    # ---- helpers
    def new(self, *shape, fill=None):
        t = torch.empty(*shape, dtype=F64, device=self.state.device)
        if fill is not None:
            t.fill_(fill)
        self.keep.append(t)
        return t

    def keep_tensor(self, t):
        """Keep a tensor alive for the lifetime of the plan (kernels hold raw device pointers) and return it."""
        self.keep.append(t)
        return t

    def rng_site(self):
        self.n_sites += 1
        return K.rng(seed=self.seed, sweep=self.sweep_counter, chain_offset=self.chain_offset, site=self.n_sites)

    def ctx(self, sampler):
        """Per-sampler persistent context (RNG site, injected draws, probes) — compile() may run more than once."""
        c = self.__dict__.setdefault("_ctx", {})
        return c.setdefault(id(sampler), {})

    def debug_tensor(self, value, size):
        """Injected draws -> (device tensor [n_sweeps, C, size], sweep stride).  Accepts [size], [C,size],
        [n_sweeps,C,size] (trailing singleton dims ignored)."""
        C = self.state.n_chains
        a = np.asarray(value, dtype=np.float64)
        if a.size == size:
            a = np.broadcast_to(a.reshape(1, 1, size), (1, C, size))
        elif a.size == C * size:
            a = a.reshape(1, C, size)
        else:
            if a.size % (C * size) != 0:
                raise ValueError(f"injected draws of size {a.size} do not match n_chains={C} x size={size}")
            a = a.reshape(-1, C, size)
        t = torch.from_numpy(np.array(a, dtype=np.float64, order="C", copy=True)).to(self.state.device)
        self.keep.append(t)
        return t, (C * size if a.shape[0] > 1 else 0)

    def emit(self, fn, label, fop=None):
        """Append a launch.  `fop` (optional): a callable returning the omc_fop_t descriptor of the same operation, which
        makes it eligible for fusion with its neighbours (fuse_small_ops)."""
        self.ops.append((label, fn))
        if fop is not None:
            self.__dict__.setdefault("_fops", {})[id(fn)] = (fn, fop)

    def add_quantity(self, q: Quantity):
        self.quantities[q.name] = q
        self.valid[q.name] = False

    def require(self, qname):
        if not self.valid[qname]:
            q = self.quantities[qname]
            q.compute()
            self.valid[qname] = True
            for s in q.siblings:
                self.valid[s] = True

    def wrote(self, param):
        for q in self.quantities.values():
            if param in q.deps:
                self.valid[q.name] = False


def fuse_small_ops(plan: Plan, ops: list) -> list:
    """Replace every run of >= 2 consecutive fusable launches of `ops` by one omc_fused_small launch (same order)."""
    if not FUSE_SMALL:
        return ops
    fops = plan.__dict__.get("_fops", {})
    C = plan.state.n_chains
    out, run = [], []

    def flush():
        while run:
            chunk = run[:K._cabi.FUSED_MAX_OPS]
            del run[:K._cabi.FUSED_MAX_OPS]
            if len(chunk) == 1:
                out.append(chunk[0][:2])
            else:
                label = "fused[" + " + ".join(lbl for lbl, _, _ in chunk) + "]"
                out.append((label, K.fused_small(C, [mk() for _, _, mk in chunk])))

    for label, fn in ops:
        hit = fops.get(id(fn))
        if hit is not None and hit[0] is fn:
            run.append((label, fn, hit[1]))
        else:
            flush()
            out.append((label, fn))
    flush()
    return out


# ---------------------------------------------------------------------------------------------- replicated responses
REP_TAG = "__replicates__"


def unreplicate(dists, state: dict, sampled=frozenset()):
    """Rewrite Normal distributions whose DATA response holds replicates in its columns (the reference's (dim, n_rep)
    convention, distribution.py:8-10; its introductory examples 1 and 2) into the single-column form the device path
    runs:  y (dim x n_rep) ~ N(h, Q) for every column, h an Identity mean  ==>  vec(y) ~ N(A h, I_n_rep (x) Q) with A the
    n_rep stacked identities -- the same density, now a LinearCombination mean with a diagonal precision, i.e. the
    regression record / Normal-linear term that exist already.  A LinearCombination mean X beta (one value per row, the
    same for every replicate) is handled the same way with X stacked n_rep times.  Applies when the response is not
    sampled, the mean is an Identity parameter of one column or a LinearCombination over data designs, and the
    precision matrix is not sampled and diagonal (always so for dim = 1).
    Returns (dists', state', changed); the inputs are left untouched."""
    from openmcmc_b200.distribution.location_scale import Normal

    out, new_state, changed = [], state, False
    for d in dists:
        y = state.get(d.response) if type(d) is Normal else None
        linear = y is not None and type(d.mean) is LinearCombination   # (round 2) mean X beta: the design is stacked n_rep times
        ok = (y is not None and d.response not in sampled and isinstance(y, np.ndarray) and y.ndim == 2 and y.shape[1] > 1
              and (linear or type(d.mean) is Identity) and d.domain_response_lower is None
              and d.domain_response_upper is None)
        if ok:
            dim, n_rep = y.shape
            if linear:
                for prm, xname in d.mean.form.items():
                    X = state.get(xname)
                    ok = (ok and X is not None and xname not in sampled and isinstance(X, np.ndarray) and X.ndim == 2
                          and X.shape[0] == dim)
            else:
                m = state.get(d.mean.form)
                ok = m is not None and not sparse.issparse(m) and not isinstance(m, torch.Tensor) and np.size(m) == dim
        if ok:
            if isinstance(d.precision, ScaledMatrix):
                pname, sname = d.precision.matrix, d.precision.scalar
            elif type(d.precision) is Identity:
                pname, sname = d.precision.form, None
            else:
                pname = None
            ok = pname is not None and pname not in sampled and pname in state and not isinstance(state[pname], torch.Tensor)
        if ok:
            P = state[pname]
            Pd = P.toarray() if sparse.issparse(P) else np.atleast_2d(np.asarray(P, dtype=np.float64))
            ok = Pd.shape == (dim, dim) and not np.any(Pd - np.diag(np.diag(Pd)))
        if not ok:
            out.append(d)
            continue
        if not changed:
            new_state, changed = dict(state), True
        tag = f"{REP_TAG}{d.response}:"
        new_state[d.response] = np.ascontiguousarray(np.asarray(y, dtype=np.float64).T).reshape(-1, 1)   # column after column
        new_state[tag + "P"] = sparse.diags([np.tile(np.diag(Pd), n_rep)], [0], format="csc")
        if linear:
            form2 = {}
            for prm, xname in d.mean.form.items():
                new_state[tag + "X:" + xname] = np.tile(np.asarray(state[xname], dtype=np.float64), (n_rep, 1))
                form2[prm] = tag + "X:" + xname
            mean2 = LinearCombination(form=form2)
        else:
            new_state[tag + "A"] = np.tile(np.eye(dim), (n_rep, 1))
            mean2 = LinearCombination(form={d.mean.form: tag + "A"})
        prec2 = ScaledMatrix(matrix=tag + "P", scalar=sname) if sname else Identity(tag + "P")
        out.append(Normal(d.response, mean=mean2, precision=prec2))
    return out, new_state, changed


# ---------------------------------------------------------------------------------------------- matching helpers
def _scalar_and_matrix(precision):
    """(matrix_name, scalar_name|None) of a precision Parameter."""
    if isinstance(precision, ScaledMatrix):
        return precision.matrix, precision.scalar
    if isinstance(precision, Identity):
        return precision.form, None
    raise PlanError(f"precision parameter {type(precision).__name__} is not supported by the device path")


def _mat_kind(arr: DevArray):
    return {"eye": K.MAT_EYE, "diag": K.MAT_DIAG, "dense": K.MAT_DENSE}[arr.kind]


def ensure_matrix(state: DeviceState, host_state: dict, name: str) -> DevArray:
    """(Re-)upload `name` as a structured square matrix (eye/diag/tridiag/dense)."""
    arr = state.arrays.get(name)
    if arr is not None and (arr.is_matrix or arr.kind != "dense" or arr.rows != arr.cols or arr.per_chain):
        return arr
    return state.put(name, host_state[name], as_matrix=True)


class RegressionLikelihood:
    """y ~ N(X beta (+ nothing else), (tau * W)^-1) with W = I or diag: owner of the fused pass (omc_reg_pass)."""

    def __init__(self, plan: Plan, host_state, dist, param, data_only=False):
        """data_only: the pass runs with beta = NULL, so the record holds rss = y'Wy and depends on the data alone (the
        form the Normal-linear MH term consumes: S(f) = y'Wy - 2 g'f + f'G f for any candidate f)."""
        st = plan.state
        self.plan = plan
        self.dist = dist
        self.param = param
        self.data_only = data_only
        form = dist.mean.form
        if param not in form:
            raise PlanError(f"'{param}' is not a term of the mean of '{dist.response}'")
        # other terms of the mean: the pass runs on y - predictor_conditional(exclude param) (sampler.py:188-192)
        self.others = [(st[pref], st[prm], bool((getattr(dist.mean, "transform", None) or {}).get(prm, False)), prm, pref)
                       for prm, pref in form.items() if prm != param]
        if len(self.others) > 4:
            raise PlanError("LinearCombination means with more than 5 terms are not supported by the device path")
        if data_only and self.others:
            raise PlanError("MH through a linear Normal mean supports a single-term LinearCombination")
        self.X = st[form[param]]
        self.y = st[dist.response]
        self.beta = st[param]
        for Xo, tho, _, prm, _ in self.others:
            if Xo.kind != "dense" or tho.cols != 1 or Xo.rows != self.X.rows:
                raise PlanError(f"unsupported term '{prm}' in the mean of '{dist.response}'")
        if self.y.cols != 1 or self.beta.cols != 1:
            raise PlanError("replicated responses (n_rep > 1) are not supported by the regression device path yet")
        self.n, self.p = self.X.rows, self.X.cols
        if self.p > 512:
            raise PlanError(f"p={self.p} > 512 regression coefficients are not supported by the device path")
        mname, self.scalar = _scalar_and_matrix(dist.precision)
        W = ensure_matrix(st, host_state, mname)
        if W.kind not in ("eye", "diag"):
            raise PlanError("the regression likelihood precision must be (a scalar times) the identity or a diagonal")
        self.W = W
        C = st.n_chains
        self.rec = self.p * self.p + self.p + 2
        self.stats = plan.new(C, self.rec, fill=0.0)
        ns, ws = K.reg_pass_workspace(C, self.n, self.p)
        self.work = plan.new(max(ws, 1))
        self.y_eff = plan.new(C, self.n) if self.others else None
        deps_other = frozenset(x for _, _, _, prm, pref in self.others for x in (prm, pref))
        deps_data = frozenset({form[param], dist.response, mname}) | deps_other
        tag = ("data:" if data_only else "") + (f"{param}|" if self.others else "")
        self.q_gg = f"gram[{tag}{dist.response}]"
        self.q_rss = f"rss[{tag}{dist.response}]"
        plan.add_quantity(Quantity(self.q_gg, deps_data, self._emit_pass, (self.q_rss,)))
        plan.add_quantity(Quantity(self.q_rss, deps_data if data_only else deps_data | {param}, self._emit_rss,
                                   (self.q_gg,)))
        ws = K.nn_dense_workspace(C, self.p)
        self.dense_ws = plan.new(ws) if ws else None
        # re-centred statistics: only when G | g | centre depend on data alone (nothing they read is sampled)
        self.center = None
        if (RECENTER and plan.recenter and CACHE_DATA_ONLY and not data_only and not self.others
                and not (deps_data & set(st.per_chain_names))):
            self.center = plan.new(C, 2 * self.p + 2, fill=0.0)     # beta_hat | c0 | rss0 | cnt
            self.q_center = f"center[{dist.response}]"
            plan.add_quantity(Quantity(self.q_center, deps_data, self._emit_center))
        self.deps_data = deps_data
        self.eig = None

    def _emit_center(self):
        """Prologue only: centre beta_hat = (G with a 1e-12 relative diagonal jitter)^-1 g, then ONE explicit-residual
        stream r0 = y - X beta_hat and the fused pass on (X, r0): c0 = X'W r0, rss0 = r0'W r0."""
        plan, st = self.plan, self.plan.state
        C, n, p = st.n_chains, self.n, self.p
        X, y, W = self.X, self.y, self.W
        w = W.data if W.kind == "diag" else None
        zero = plan.new(1, fill=0.0)
        plan.require(self.q_gg)

        def launch():
            dev = st.device
            beta_hat = torch.empty(C, p, dtype=F64, device=dev)
            K.nn_dense_draw(C, p, self.stats, K.vec(None), K.MAT_EYE, K.vec(None), K.vec(zero), K.vec(None), beta_hat,
                            K.rng(), solve_only=True, ridge_rel=1e-12, workspace=self.dense_ws)
            r0 = torch.empty(C, n, dtype=F64, device=dev)
            K.linear_predictor(C, n, [(X.vec(), K.vec(beta_hat, p), p, False)], r0, residual_of=y.vec())
            scratch = torch.empty(C, self.rec, dtype=F64, device=dev)
            K.reg_pass(X.data, r0, w, None, scratch, self.work, C, n, p, x_shared=not X.per_chain, y_shared=False,
                       w_shared=True)
            self.center[:, :p].copy_(beta_hat)                        # plumbing: the kernels did the arithmetic
            self.center[:, p:].copy_(scratch[:, p * p:])

        plan.emit(launch, "reg_center")

    def eigen_record(self, P0, mu0, prior_names):
        """The eigen record M | D | h | m | u_hat | k of the element-wise dense draw (omc.h: omc_nn_eigen_prep), for the
        prior precision P0 (eye or diagonal DevArray) and mean mu0 named in prior_names.  Data only, like the centre it
        reads: computed in the prologue.  Returns (record [C, p*p + 5p], quantity name)."""
        if self.eig is None:
            self.eig = self.plan.new(self.plan.state.n_chains, K.eigen_record_len(self.p), fill=0.0)
            self.q_eig = f"eigen[{self.dist.response}]"
            self.plan.add_quantity(Quantity(self.q_eig, self.deps_data | frozenset(prior_names),
                                            lambda: self._emit_eigen(P0, mu0)))
        return self.eig, self.q_eig

    def _emit_eigen(self, P0, mu0):
        plan = self.plan
        plan.require(self.q_center)
        C, p = plan.state.n_chains, self.p

        def launch():
            K.nn_eigen_prep(C, p, self.stats, _mat_kind(P0), P0.vec(), mu0.vec(), self.center, self.eig)

        plan.emit(launch, "nn_eigen_prep")

    def rss_ptr(self):
        return self.stats.data_ptr() + 8 * (self.p * self.p + self.p)

    def _emit_rss(self):
        """rss is stale.  While G | g (data only) are still valid, X is streamed for the residual alone (omc_reg_rss,
        HBM-bound); otherwise the full pass refreshes the whole record."""
        if self.data_only or not self.plan.valid[self.q_gg] or not CACHE_DATA_ONLY:
            return self._emit_pass()
        return self._emit_pass(rss_only=True)

    def _emit_pass(self, rss_only=False):
        C, n, p = self.plan.state.n_chains, self.n, self.p
        X, y, W, beta, stats, work = self.X, self.y, self.W, self.beta, self.stats, self.work
        w = W.data if W.kind == "diag" else None
        beta_data = None if self.data_only else beta.data
        others, y_eff = self.others, self.y_eff

        kernel = K.reg_rss if rss_only else K.reg_pass

        def launch():
            if others:
                K.linear_predictor(C, n, [(Xo.vec(), tho.vec(), Xo.cols, tr) for Xo, tho, tr, _, _ in others], y_eff,
                                   residual_of=y.vec())
                kernel(X.data, y_eff, w, beta_data, stats, work, C, n, p, x_shared=not X.per_chain, y_shared=False,
                       w_shared=True)
                return
            kernel(X.data, y.data, w, beta_data, stats, work, C, n, p, x_shared=not X.per_chain,
                   y_shared=not y.per_chain, w_shared=True)

        self.plan.emit(launch, "reg_rss" if rss_only else "reg_pass")

    # views into the record
    def rss_vec(self):
        return K.vec((self.stats[:, self.p * self.p + self.p:], self.rec))

    def cnt_vec(self):
        return K.vec((self.stats[:, self.p * self.p + self.p + 1:], self.rec))


class MixtureNormal:
    """x_i ~ N(mu[z_i], 1/tau[z_i]) (MixtureParameterVector mean, MixtureParameterMatrix precision): owner of the
    per-component sufficient statistics, the regression-format record for a NormalNormal update of mu, and the gathers
    mu[z], tau[z] a NormalNormal update of x uses as its prior.  ref: parameter.py:377-538, sampler.py:272-355."""

    def __init__(self, plan: Plan, host_state, dist):
        from openmcmc_b200.parameter import MixtureParameterMatrix, MixtureParameterVector

        if not isinstance(dist.mean, MixtureParameterVector) or not isinstance(dist.precision, MixtureParameterMatrix):
            raise PlanError("a mixture Normal needs a MixtureParameterVector mean and a MixtureParameterMatrix precision")
        if dist.mean.allocation != dist.precision.allocation:
            raise PlanError("mixture mean and precision must share their allocation parameter")
        st = plan.state
        self.plan, self.dist = plan, dist
        self.names = (dist.response, dist.mean.param, dist.precision.param, dist.mean.allocation)
        self.x, self.mu, self.tau, self.z = (st[nm] for nm in self.names)
        if self.x.cols != 1:
            raise PlanError("replicated mixture responses (n_rep > 1) are not supported by the device path")
        if not self.z.per_chain:
            self.z = st.put(dist.mean.allocation, host_state[dist.mean.allocation], per_chain=True)
        self.n, self.K = self.x.rows, self.mu.size
        if self.tau.size != self.K or self.K > 64:
            raise PlanError(f"mixture with {self.mu.size} means / {self.tau.size} precisions (at most 64 components)")
        C = st.n_chains
        self.rec = self.K * self.K + self.K + 2
        self.stats = plan.new(C, self.K, 4, fill=0.0)
        self.record = plan.new(C, self.rec, fill=0.0)
        self.g_mu, self.g_tau = plan.new(C, self.n), plan.new(C, self.n)
        self.qname = f"mixture[{dist.response}]"
        plan.add_quantity(Quantity(self.qname, frozenset(self.names), self._emit))

    def _emit(self):
        C = self.plan.state.n_chains

        def launch():
            K.mixture_stats(C, self.n, self.K, self.x.vec(), self.mu.vec(), self.tau.vec(), self.z.data, self.stats,
                            record=self.record, gather_mu=self.g_mu, gather_tau=self.g_tau)

        self.plan.emit(launch, f"mixture_stats[{self.dist.response}]")

    def emit_log_p(self, out, acc):
        """Normal log-density of x under the current allocation (fresh pass: log_post runs after the sweep)."""
        C = self.plan.state.n_chains
        scratch = self.plan.new(C, self.K, 4)

        def launch():
            K.mixture_stats(C, self.n, self.K, self.x.vec(), self.mu.vec(), self.tau.vec(), self.z.data, scratch,
                            logp=out, accumulate=acc)

        self.plan.emit(launch, f"logp_mixture[{self.dist.response}]")


def get_mixture(plan: Plan, host_state, dist) -> MixtureNormal:
    cache = plan.__dict__.setdefault("_mixtures", {})
    if dist.response not in cache:
        cache[dist.response] = MixtureNormal(plan, host_state, dist)
    return cache[dist.response]


def compile_fitted(plan: Plan, host_state, dist, predictor: str, n_iter: int, ring: bool = False):
    """Fitted values store[response][:, it] = dist.<predictor>.predictor(state).  ref: mcmc.py:109-111.
    n_iter rows, or (ring) a ring of n_iter slabs for the streamed store."""
    st = plan.state
    C = st.n_chains
    par = getattr(dist, predictor)
    n = st[dist.response].rows
    buf = plan.new(n_iter, C, n, fill=float("nan"))
    if isinstance(par, LinearCombination):
        now = plan.new(C, n)
        terms = []
        transform = getattr(par, "transform", None) or {}
        for prm, pref in par.form.items():
            X, th = st[pref], st[prm]
            if X.kind != "dense" or th.cols != 1:
                raise PlanError("fitted values: unsupported LinearCombination term")
            terms.append((X, th, bool(transform.get(prm, False))))
        if len(terms) > 4:
            raise PlanError("fitted values: more than 4 LinearCombination terms")

        def launch():
            K.linear_predictor(C, n, [(X.vec(), th.vec(), X.cols, tr) for X, th, tr in terms], now)
            K.store_copy(now, buf, C * n, plan.iter_counter, n_iter, ring=ring)

        plan.emit(launch, f"fitted[{dist.response}]")
    elif isinstance(par, Identity):
        src = st[par.form]
        if not src.per_chain:
            src = st.put(par.form, src.data, per_chain=True)

        def launch():
            K.store_copy(src.data, buf, C * n, plan.iter_counter, n_iter, ring=ring)

        plan.emit(launch, f"fitted[{dist.response}]")
    else:
        raise PlanError(f"fitted values for {type(par).__name__} are not supported on the device")
    return buf


def as_chain_tensor(value, n_chains, size, device):
    """Injected draws: accept [size], [size,1], [C,size] or [C,size,1]; broadcast over chains."""
    a = np.asarray(value, dtype=np.float64)
    if a.size == size:
        a = np.broadcast_to(a.reshape(1, size), (n_chains, size))
    else:
        a = a.reshape(n_chains, size)
    return torch.as_tensor(np.ascontiguousarray(a)).to(device)


def get_regression(plan: Plan, host_state, lik, param, data_only=False) -> RegressionLikelihood:
    cache = plan.__dict__.setdefault("_regressions", {})
    key = (lik.response, data_only) if data_only else lik.response
    if isinstance(lik.mean, LinearCombination) and len(lik.mean.form) > 1:
        key = (lik.response, param, data_only)      # one record per term of a multi-term mean
    if key not in cache:
        cache[key] = RegressionLikelihood(plan, host_state, lik, param, data_only=data_only)
    return cache[key]


def get_quadratic_form(plan: Plan, host_state, nrm):
    """Quadratic form r' P r (P un-scaled) and #(diag P > 0) of a Normal distribution's residual.

    Returns (ss_vec_fn, cnt_vec_fn, quantity_name).  ref: sampler.py:275-284.
    """
    st = plan.state
    from openmcmc_b200 import gmrf_plan

    fields = gmrf_plan._fields(plan)
    if fields and (nrm.response in fields or gmrf_plan._quick_mean_name(nrm) in fields):
        mname, _ = _scalar_and_matrix(nrm.precision)
        P = ensure_matrix(st, host_state, mname)
        if nrm.response in fields or gmrf_plan._identity_mean_of(plan, host_state, nrm) in fields:
            key = nrm.response
            cache = plan.__dict__.setdefault("_quadforms", {})
            if key not in cache:
                cache[key] = gmrf_plan.long_quadratic_form(plan, host_state, nrm, P, None, None)
            return cache[key]
    if isinstance(nrm.mean, LinearCombination):
        params = list(nrm.mean.form.keys())
        rl = get_regression(plan, host_state, nrm, params[0])
        return rl.rss_vec, rl.cnt_vec, rl.q_rss
    if not isinstance(nrm.mean, Identity):
        raise PlanError(f"unsupported Normal mean {type(nrm.mean).__name__}")
    cache = plan.__dict__.setdefault("_quadforms", {})
    key = nrm.response
    if key in cache:
        return cache[key]
    mname, _ = _scalar_and_matrix(nrm.precision)
    P = ensure_matrix(st, host_state, mname)
    x, mu = st[nrm.response], st[nrm.mean.form]
    C = st.n_chains
    if x.cols != 1:
        raise PlanError("replicated responses (n_rep > 1) are not supported by the device quadratic form yet")
    if P.kind == "tridiag" or x.rows > 4096:
        out = gmrf_plan.long_quadratic_form(plan, host_state, nrm, P, x, mu)
        cache[key] = out
        return out
    ss, cnt = plan.new(C), plan.new(C)
    qname = f"quad[{nrm.response}]"
    p = x.rows

    def compute():
        def launch():
            K.quadform(C, p, x.vec(), mu.vec(), _mat_kind(P), P.vec(), ss, cnt)

        fop = (lambda: K.fop_quadform(C, p, x.vec(), mu.vec(), _mat_kind(P), P.vec(), ss, cnt)) \
            if P.kind in ("eye", "diag") and p <= 512 else None
        plan.emit(launch, f"quadform[{nrm.response}]", fop=fop)

    plan.add_quantity(Quantity(qname, frozenset({nrm.response, nrm.mean.form, mname}), compute))
    out = (lambda: K.vec(ss, 1), lambda: K.vec(cnt, 1), qname)
    cache[key] = out
    return out


def logdet_of(plan: Plan, P: DevArray):
    """log|P| of a constant structured matrix, computed once on the device at plan time (None => 0)."""
    if P.kind == "eye":
        return None
    C = plan.state.n_chains
    out = plan.new(1 if not P.per_chain else C)
    if P.kind == "diag":
        K.sum_log(P.data, P.rows, out)
    elif P.kind == "dense":
        K.logdet_dense(P.data, P.rows, out)
    else:
        from openmcmc_b200 import gmrf_plan

        gmrf_plan.tridiag_logdet(plan, P, out)
    return out


def lognormal_shim(plan: Plan, dist):
    """A LogNormal whose response y is DATA, seen from its mean / precision parameters, is the Normal of log(y) with the
    same mean and precision, minus the constant sum(log y) (location_scale.py:296-303; mean-parameter branch of the
    gradient / Hessian :344-347, :401-404).  Returns (Normal on the derived state entry `__log[y]`, -sum(log y) per chain).
    The log of the data is taken once, on the device, when the plan is built."""
    from openmcmc_b200.distribution.location_scale import Normal

    st = plan.state
    if dist.response in st.per_chain_names:
        raise PlanError(f"LogNormal '{dist.response}' is sampled and enters through its mean: not supported on the device")
    shims = plan.__dict__.setdefault("_lognormal_shims", {})
    if dist.response not in shims:
        y = st[dist.response]
        name = f"__log[{dist.response}]"
        logy = torch.empty_like(y.data)
        K.log_elements(y.data, logy)
        st.put(name, logy)
        m = st.n_chains if y.per_chain else 1
        s = plan.new(m)
        K.sum_log(y.data, y.size, s)
        const = plan.new(st.n_chains)
        K.combine(st.n_chains, 1, [K.vec(s, 1 if y.per_chain else None)], [K.vec(plan.new(1, fill=-1.0))], const)
        shims[dist.response] = (name, const)
    name, const = shims[dist.response]
    return Normal(name, mean=dist.mean, precision=dist.precision), const


def compile_log_post(plan: Plan, host_state, model, out, accumulate_first=False):
    """Emit kernels accumulating model.log_p(state) per chain into `out` [C].  ref: mcmc.py:108, model.py:57-70."""
    from openmcmc_b200.distribution.distribution import Categorical, Gamma, Poisson, Uniform
    from openmcmc_b200.distribution.location_scale import LogNormal, Normal, NullDistribution
    from openmcmc_b200.parameter import MixtureParameterMatrix

    st = plan.state
    C = st.n_chains
    first = not accumulate_first
    for dist in model.values():
        acc = 0 if first else 1
        if isinstance(dist, NullDistribution):
            continue
        transformed = isinstance(dist, Normal) and any((getattr(dist.mean, "transform", None) or {}).values())
        if (isinstance(dist, LogNormal) and not isinstance(dist.mean, Identity)
                and dist.response not in st.per_chain_names):
            # data response, structured mean: Normal of log(y) minus sum(log y)
            from openmcmc_b200.model import Model

            shim, const = lognormal_shim(plan, dist)
            compile_log_post(plan, host_state, Model([shim]), out, accumulate_first=not first)
            one = plan.new(1, fill=1.0)

            def launch(const=const, one=one):
                K.combine(C, 1, [K.vec(out, 1), K.vec(const, 1)], [K.vec(one), K.vec(one)], out)

            plan.emit(launch, f"logp_lognormal_jacobian[{dist.response}]")
        elif isinstance(dist, LogNormal) or transformed:
            # no dedicated kernel: the distribution as a one-term MH model of its response (LogNormal) or of the
            # transformed coefficient vector (Normal with a LinearCombinationWithTransform mean)
            from openmcmc_b200 import devdist
            from openmcmc_b200.model import Model

            if transformed and len(dist.mean.form) != 1:
                raise PlanError("log_post: LinearCombinationWithTransform means with more than one term are not supported")
            prm = dist.response if isinstance(dist, LogNormal) else next(iter(dist.mean.form))
            tm, _ = devdist.build_terms(plan, host_state, Model([dist]), prm)
            x = st[prm]

            def launch(tm=tm, x=x, acc=acc):
                K.mh_logp(tm, x.data, out, accumulate=acc)

            plan.emit(launch, f"logp_terms[{dist.response}]")
        elif isinstance(dist, Normal) and isinstance(dist.precision, MixtureParameterMatrix):
            get_mixture(plan, host_state, dist).emit_log_p(out, acc)
        elif isinstance(dist, Categorical):
            z, prob = st[dist.response], st[dist.prob.form]
            if z.cols != 1:
                raise PlanError("log_post: replicated Categorical responses are not supported on the device")
            if not z.per_chain:
                z = st.put(dist.response, host_state[dist.response], per_chain=True)
            kk = prob.cols
            prob_rows = prob.rows
            if prob_rows not in (1, z.rows):
                raise PlanError("Categorical: prob must have 1 or n rows")

            def launch(z=z, prob=prob, kk=kk, prob_rows=prob_rows, acc=acc):
                K.logp_categorical(C, z.rows, kk, z.data, prob.vec(), prob_rows, out, acc)

            plan.emit(launch, f"logp_categorical[{dist.response}]")
        elif isinstance(dist, Normal):
            mname, sname = _scalar_and_matrix(dist.precision)
            ss_vec, _, qname = get_quadratic_form(plan, host_state, dist)
            P = ensure_matrix(st, host_state, mname)
            logdet = logdet_of(plan, P)
            scal = st[sname] if sname else None
            dim = st[dist.response].rows
            plan.require(qname)

            def nargs(dim=dim, ss_vec=ss_vec, scal=scal, logdet=logdet, acc=acc):
                return (C, dim, ss_vec(), scal.vec() if scal else K.vec(None),
                        K.vec(logdet) if logdet is not None else K.vec(None), out, acc)

            plan.emit((lambda nargs=nargs: K.logp_normal_ss(*nargs())), f"logp_normal[{dist.response}]",
                      fop=(lambda nargs=nargs: K.fop_logp_normal_ss(*nargs())))
            if dist.domain_response_lower is not None or dist.domain_response_upper is not None:
                # -inf outside the domain; the truncation normaliser is ignored (location_scale.py:148-151,164-165)
                x = st[dist.response]

                def bound(v, size=x.size):
                    if v is None:
                        return K.vec(None), 1
                    t = plan.keep_tensor(torch.as_tensor(np.asarray(v, dtype=np.float64).reshape(-1)).to(st.device))
                    if t.numel() not in (1, size):
                        raise ValueError(f"domain bound of size {t.numel()} for a response of size {size}")
                    return K.vec(t), int(t.numel())

                (lo_v, lo_n), (hi_v, hi_n) = bound(dist.domain_response_lower), bound(dist.domain_response_upper)

                def launch(x=x, lo_v=lo_v, lo_n=lo_n, hi_v=hi_v, hi_n=hi_n):
                    K.logp_domain(C, x.size, x.vec(), lo_v, lo_n, hi_v, hi_n, out)

                plan.emit(launch, f"logp_domain[{dist.response}]")
        elif isinstance(dist, Gamma):
            x = st[dist.response]
            if not isinstance(dist.shape, Identity) or not isinstance(dist.rate, Identity):
                raise PlanError("log_post: Gamma with non-Identity shape/rate is not supported on the device yet")
            sh, rt = st[dist.shape.form], st[dist.rate.form]

            def gargs(x=x, sh=sh, rt=rt, acc=acc):
                return (C, x.size, x.vec(), sh.vec(), sh.size, rt.vec(), rt.size, out, acc)

            plan.emit((lambda gargs=gargs: K.logp_gamma(*gargs())), f"logp_gamma[{dist.response}]",
                      fop=(lambda gargs=gargs: K.fop_logp_gamma(*gargs())) if x.size <= 256 else None)
        elif isinstance(dist, Poisson):
            k = st[dist.response]
            if not isinstance(dist.rate, Identity):
                raise PlanError("log_post: Poisson with non-Identity rate is not supported on the device yet")
            rt = st[dist.rate.form]

            def pargs(k=k, rt=rt, acc=acc):
                return (C, k.size, k.vec(), rt.vec(), rt.size, out, acc)

            plan.emit((lambda pargs=pargs: K.logp_poisson(*pargs())), f"logp_poisson[{dist.response}]",
                      fop=(lambda pargs=pargs: K.fop_logp_poisson(*pargs())) if k.size <= 256 else None)
        elif isinstance(dist, Uniform):
            x = st[dist.response]
            rng_ = np.broadcast_to(dist.domain_response_upper - dist.domain_response_lower, (x.rows, 1))
            value = -float(np.sum(np.log(rng_))) * x.cols

            plan.emit((lambda value=value, acc=acc: K.logp_const(value, C, out, acc)), f"logp_uniform[{dist.response}]",
                      fop=(lambda value=value, acc=acc: K.fop_logp_const(value, C, out, acc)))
        else:
            raise PlanError(f"log_post: distribution {type(dist).__name__} is not supported on the device")
        first = False
    if first:

        def launch():
            K.logp_const(0.0, C, out, 0)

        plan.emit(launch, "logp_zero")
