"""MCMCSampler base class and the conjugate samplers NormalNormal / NormalGamma.  ref: sampler/sampler.py:37-288

The classes keep the reference's constructor signatures and `.sample(state) -> state` contract.  Numerically they are
*plan fragments*: `compile(plan, host_state)` appends the CUDA kernel launches of one update to the sweep plan
(engine.Plan); `.sample()` on a host dict compiles and runs a one-sampler plan on the device (n_chains = 1).
MixtureAllocation (SURVEY §8 f2) draws the allocations of a mixture Normal; NormalGamma / NormalNormal understand the
MixtureParameterVector / MixtureParameterMatrix parameters of that Normal.
"""

from abc import ABC, abstractmethod
from dataclasses import dataclass
from typing import Union

import numpy as np

from openmcmc_b200 import engine
from openmcmc_b200 import kernels as K
from openmcmc_b200.distribution.location_scale import Normal
from openmcmc_b200.model import Model
from openmcmc_b200.parameter import (
    Identity,
    LinearCombination,
    MixtureParameterMatrix,
    MixtureParameterVector,
    ScaledMatrix,
)


@dataclass
class MCMCSampler(ABC):
    """ref: sampler.py:37-118"""

    param: str
    model: Model
    max_variable_size: Union[int, tuple, None] = None

    def __post_init__(self):
        self.model = self.model.conditional(self.param)

    def sample(self, current_state: dict, debug_draws: dict = None) -> dict:
        """Generate the next sample of self.param on the device and return the updated state dict.

        `debug_draws` (extension) injects the reference's random streams, e.g. {"z": ...} for NormalNormal,
        {"g": ...} for NormalGamma (standard-gamma variates), mirroring the reference tests' rvs patches.
        """
        from openmcmc_b200 import hostcalls

        return hostcalls.sample_once(self, current_state, debug_draws)

    @abstractmethod
    def compile(self, plan: "engine.Plan", host_state: dict, debug_draws: dict = None):
        """Append this sampler's kernel launches to the sweep plan."""

    def init_store(self, current_state: dict, store: dict, n_iterations: int) -> dict:
        """ref: sampler.py:69-87"""
        if self.max_variable_size is None:
            store[self.param] = np.full(shape=(np.size(current_state[self.param]), n_iterations), fill_value=np.nan)
        elif isinstance(self.max_variable_size, tuple):
            store[self.param] = np.full(shape=self.max_variable_size + (n_iterations,), fill_value=np.nan)
        else:
            store[self.param] = np.full(shape=(self.max_variable_size, n_iterations), fill_value=np.nan)
        return store

    def store(self, current_state: dict, store: dict, iteration: int) -> dict:
        """ref: sampler.py:89-118 (host copy of one column; the device path stores with omc_store_copy instead)"""
        current_param = np.asarray(current_state[self.param])
        if self.max_variable_size is None:
            store[self.param][:, [iteration]] = current_param.reshape(-1, 1)
        elif isinstance(self.max_variable_size, tuple):
            index_list = [np.arange(current_param.shape[dim], dtype=int) for dim in range(current_param.ndim)]
            index_list.append(np.array([iteration]))
            store[self.param][np.ix_(*index_list)] = current_param.reshape(current_param.shape + (1,))
        else:
            store[self.param][range(current_param.size), [iteration]] = current_param.flatten()
        return store


@dataclass
class NormalNormal(MCMCSampler):
    """Normal-Normal conjugate update.  ref: sampler.py:121-207

    Device paths (chosen from the model structure at compile time):
      * dense   : one Normal likelihood with mean X @ param (LinearCombination), diagonal/identity response precision,
                  any prior precision up to p = 512            -> omc_reg_pass + omc_nn_dense_draw
      * banded  : one Normal likelihood with mean = param (Identity), diagonal/identity response precision, tridiagonal
                  prior precision (temporal GMRF)              -> omc_tridiag_nn_draw
    Truncated priors (domain_response_lower / upper on the Normal prior; sampler.py:196-205 ->
    gmrf.gibbs_canonical_truncated_normal, SURVEY §8 f3) are supported on the dense path up to p = 512: the draw
    becomes one coordinate-wise truncated-normal Gibbs scan from the current value.  `debug_draws={"u": ...}` injects
    the uniforms behind the reference's truncnorm.rvs calls.
    """

    def __post_init__(self):
        super().__post_init__()
        self._is_response = {key: key == self.param for key in self.model.keys()}

    def compile(self, plan, host_state, debug_draws=None):
        prior = self.model[self.param]
        if not isinstance(prior, Normal):
            raise engine.PlanError("NormalNormal needs a Normal prior on the sampled parameter")
        liks = [d for k, d in self.model.items() if not self._is_response[k]]
        if not liks or not all(isinstance(d, Normal) for d in liks):
            raise engine.PlanError("the device NormalNormal needs Normal likelihood terms (and at least one)")
        from openmcmc_b200 import gmrf_plan

        if (len(liks) == 1 and not isinstance(prior.precision, MixtureParameterMatrix)
                and gmrf_plan.is_gmrf_update(plan, host_state, self.param, prior, liks[0])):
            if prior.domain_response_lower is not None or prior.domain_response_upper is not None:
                raise engine.PlanError("a truncated prior on the tridiagonal (GMRF) path is not supported: the "
                                       "coordinate-wise scan of gmrf.py:201-266 is sequential over 1e6 elements")
            return gmrf_plan.compile_normal_normal_identity(self, plan, host_state, prior, liks[0], debug_draws)
        # dense path: every likelihood term contributes a regression record (sampler.py:179-192).  A term whose mean is
        # the parameter itself (Identity) is the regression on the p x p identity.
        liks = [self._as_regression(plan, host_state, d) for d in liks]
        if len(liks) == 1:
            return self._compile_dense(plan, host_state, prior, liks[0], debug_draws)
        return self._compile_dense(plan, host_state, prior, liks[0], debug_draws,
                                   source=self._combined_source(plan, host_state, liks))

    def _as_regression(self, plan, host_state, lik):
        """The likelihood as Normal(y | X param + ..., .): LinearCombination means pass through, an Identity mean on the
        sampled parameter becomes the regression on the identity matrix (b += Q_rsp y of sampler.py:187-188)."""
        if isinstance(lik.mean, LinearCombination):
            if self.param not in lik.mean.form:
                raise engine.PlanError(f"'{self.param}' is not a term of the mean of '{lik.response}'")
            return lik
        if isinstance(lik.mean, Identity) and lik.mean.form == self.param:
            p = plan.state[self.param].rows
            if p > 512:
                raise engine.PlanError(f"NormalNormal with an Identity-mean likelihood of dimension {p} and a dense "
                                       "posterior precision: only the tridiagonal (GMRF) form scales beyond 512")
            name = f"__eye{p}__"
            if name not in host_state:
                host_state[name] = np.eye(p)
            return Normal(lik.response, mean=LinearCombination(form={self.param: name}), precision=lik.precision)
        raise engine.PlanError(
            f"NormalNormal: a likelihood mean of type {type(lik.mean).__name__} is not supported by the device path")

    def _combined_source(self, plan, host_state, liks):
        """Several likelihood terms: Q and b are sums over the terms (sampler.py:179-192), so their records
        tau_l * (G_l | g_l) are added into one record per sweep (omc_combine) and the draw runs on that with tau = 1.
        The residual sums of squares stay with their own records (explicit passes: no common centre)."""
        st = plan.state
        C = st.n_chains
        rls = [engine.get_regression(plan, host_state, lik, self.param) for lik in liks]
        p = rls[0].p
        if any(r.p != p for r in rls):
            raise engine.PlanError("NormalNormal: likelihood terms with different coefficient dimensions")
        if len(rls) > 4:
            raise engine.PlanError("NormalNormal with more than 4 likelihood terms is not supported by the device path")
        rec = rls[0].rec
        comb = plan.new(C, rec, fill=0.0)
        taus = [st[r.scalar] if r.scalar else None for r in rls]

        def launch():
            K.combine(C, rec, [K.vec(r.stats, rec) for r in rls], [t.vec() if t else None for t in taus], comb)

        return dict(stats=comb, rec=rec, p=p, tau=None, require=[r.q_gg for r in rls], pre=(launch, "combine_records"))

    def _compile_dense(self, plan, host_state, prior, lik, debug_draws, source=None):
        """source (mixture-mean update): the likelihood record comes from engine.MixtureNormal instead of the regression
        pass.  A mixture PRIOR (MixtureParameterVector mean / MixtureParameterMatrix precision on the sampled vector,
        the reference's tests/test_sampler.py:113-147 model) enters as a per-chain diagonal prior tau[z] with mean mu[z]."""
        st = plan.state
        C = st.n_chains
        if source is None:
            rl = engine.get_regression(plan, host_state, lik, self.param)
            source = dict(stats=rl.stats, rec=rl.rec, p=rl.p, tau=st[rl.scalar] if rl.scalar else None, require=rl.q_gg,
                          regression=rl)
        p = source["p"]
        tau = source["tau"]
        requires = list(source["require"]) if isinstance(source["require"], (list, tuple)) else [source["require"]]
        eigen_prior = False
        if isinstance(prior.mean, MixtureParameterVector) and isinstance(prior.precision, MixtureParameterMatrix):
            mix = engine.get_mixture(plan, host_state, prior)
            requires.append(mix.qname)
            mu0_vec = lambda: K.vec(mix.g_mu, mix.n)          # noqa: E731
            P0_kind, P0_vec, lam = K.MAT_DIAG, (lambda: K.vec(mix.g_tau, mix.n)), None
        else:
            if not isinstance(prior.mean, Identity):
                raise engine.PlanError("NormalNormal: prior mean must be an Identity (or mixture) parameter")
            mu0 = st[prior.mean.form]
            pm_name, lam_name = engine._scalar_and_matrix(prior.precision)
            P0 = engine.ensure_matrix(st, host_state, pm_name)
            if P0.kind == "tridiag":
                # a GMRF prior on regression coefficients (example 4 with A != I): the posterior precision
                # lambda P + tau X'X is dense, so the prior enters the dense draw as a dense p x p matrix
                # (the tridiagonal form stays registered under its own name for the quadratic form / log-determinant)
                Pm = host_state[pm_name]
                dname = pm_name + "::dense"
                if dname not in st.arrays:
                    if Pm.shape[0] > 512:
                        raise engine.PlanError("a tridiagonal prior with a regression likelihood gives a dense posterior "
                                               f"precision: {Pm.shape[0]} > 512 coefficients are not supported")
                    st.put(dname, Pm.toarray() if engine.sparse.issparse(Pm) else np.asarray(Pm, dtype=np.float64))
                P0 = st.arrays[dname]
            lam = st[lam_name] if lam_name else None
            mu0_vec, P0_kind, P0_vec = mu0.vec, engine._mat_kind(P0), P0.vec
            # the eigenbasis of (G, P0) is data when P0 and mu0 are (and a positive diagonal P0 has one)
            eigen_prior = (P0.kind == "eye" or (P0.kind == "diag" and P0.npos == p)) and not (
                {pm_name, prior.mean.form} & set(st.per_chain_names))
        beta = st[self.param]
        ctx = plan.ctx(self)
        if "rng" not in ctx:
            ctx["rng"] = plan.rng_site()
            ctx["dz"], ctx["dz_stride"] = (None, 0)
            if debug_draws and "z" in debug_draws:
                ctx["dz"], ctx["dz_stride"] = plan.debug_tensor(debug_draws["z"], p)
            ctx["probes"] = None
            if plan.probes is not None and plan.probes.get("enable"):
                probes = {k: plan.new(C, p, p) for k in ("Q", "L")}
                probes.update({k: plan.new(C, p) for k in ("b", "mu")})
                plan.probes[self.param] = ctx["probes"] = probes
            ctx["trunc"] = None
            lo, hi = prior.domain_response_lower, prior.domain_response_upper
            if lo is not None or hi is not None:
                if p > 512:
                    raise engine.PlanError(f"NormalNormal with a truncated prior supports p <= 512 coefficients (p = {p})")
                # ref gmrf.py:236-243: missing bounds are -inf / +inf, scalars broadcast over the p coordinates
                def bound(v):
                    if v is None:
                        return K.vec(None), 1
                    t = plan.keep_tensor(engine.torch.as_tensor(np.asarray(v, dtype=np.float64).reshape(-1)).to(st.device))
                    if t.numel() not in (1, p):
                        raise ValueError(f"truncation bound of size {t.numel()} for a parameter of size {p}")
                    return K.vec(t), int(t.numel())

                (lo_v, lo_n), (hi_v, hi_n) = bound(lo), bound(hi)
                ctx["trunc"] = (lo_v, lo_n, hi_v, hi_n)
                if debug_draws and "u" in debug_draws:
                    ctx["dz"], ctx["dz_stride"] = plan.debug_tensor(debug_draws["u"], p)
        rng, dz, dz_stride, probes, trunc = ctx["rng"], ctx["dz"], ctx["dz_stride"], ctx["probes"], ctx["trunc"]
        # re-centred statistics: the draw leaves rss(beta_new) in the regression record (no pass over X; engine.RECENTER)
        rl = source.get("regression")
        centred = rl is not None and rl.center is not None and trunc is None
        if centred:
            requires.append(rl.q_center)
        # G, g, P0, mu0 and the centre all data, nothing injected or probed: the draw runs in the fixed eigenbasis of
        # (G, P0) (omc_nn_eigen_draw), a mat-vec per chain instead of a Cholesky of Q
        eigen = centred and eigen_prior and p <= K.EIGEN_MAX_P and dz is None and probes is None
        if eigen:
            eig, q_eig = rl.eigen_record(P0, mu0, (pm_name, prior.mean.form))
            requires.append(q_eig)
        for q in requires:
            plan.require(q)
        stats = source["stats"]
        center, rss_out = (rl.center, rl.rss_ptr()) if centred else (None, None)
        if rl is not None:
            workspace = rl.dense_ws
        else:
            ws = K.nn_dense_workspace(C, p)
            workspace = ctx.setdefault("workspace", plan.new(ws) if ws else None)

        if source.get("pre"):
            plan.emit(*source["pre"])

        def launch_eigen():
            K.nn_eigen_draw(C, p, eig, tau.vec() if tau else K.vec(None), lam.vec() if lam else K.vec(None), beta.data,
                            rng, status=plan.status, center=center, rss_out=rss_out, rss_stride=rl.rec)

        def launch():
            K.nn_dense_draw(
                C, p, stats, tau.vec() if tau else K.vec(None), P0_kind, P0_vec(),
                lam.vec() if lam else K.vec(None), mu0_vec(), beta.data, rng, debug_z=None if trunc else dz,
                probe_Q=probes["Q"] if probes else None, probe_b=probes["b"] if probes else None,
                probe_L=probes["L"] if probes else None, probe_mu=probes["mu"] if probes else None, status=plan.status,
                debug_sweep_stride=dz_stride, trunc=trunc, debug_u=dz if trunc else None, center=center,
                rss_out=rss_out, workspace=workspace)

        plan.emit(launch_eigen if eigen else launch, f"nn_dense_draw[{self.param}]")
        plan.wrote(self.param)
        if centred:
            plan.valid[rl.q_rss] = True


@dataclass
class NormalGamma(MCMCSampler):
    """Normal-Gamma conjugate update of a scalar precision.  ref: sampler.py:210-288

    The quadratic form r' P r comes from whichever kernel owns the Normal distribution's residual: the regression pass
    (likelihood precision), omc_quadform (small prior precision) or the tridiagonal kernels (GMRF).
    MixtureParameterMatrix precisions (the K-loop at sampler.py:281-284) are SURVEY §8 f2 ("next").
    """

    def __post_init__(self):
        super().__post_init__()
        nrm_prm = list(self.model.keys())
        nrm_prm.remove(self.param)
        self.normal_param = nrm_prm[0]
        precision = self.model[self.normal_param].precision
        if not isinstance(precision, (Identity, ScaledMatrix, MixtureParameterMatrix)):
            raise TypeError("precision must be either Identity, ScaledMatrix or MixtureParameterMatrix")

    def compile(self, plan, host_state, debug_draws=None):
        from openmcmc_b200.distribution.distribution import Gamma

        st = plan.state
        C = st.n_chains
        gam = self.model[self.param]
        nrm = self.model[self.normal_param]
        if not isinstance(gam, Gamma) or not isinstance(gam.shape, Identity) or not isinstance(gam.rate, Identity):
            raise engine.PlanError("NormalGamma needs a Gamma prior with Identity shape and rate")
        if isinstance(nrm.precision, MixtureParameterMatrix) and nrm.precision.param == self.param:
            return self._compile_mixture(plan, host_state, gam, nrm, debug_draws)
        if not isinstance(nrm.precision, ScaledMatrix) or nrm.precision.scalar != self.param:
            raise engine.PlanError("NormalGamma: the Normal precision must be ScaledMatrix(matrix, scalar=param)")
        out = st[self.param]
        if out.size != 1:
            raise engine.PlanError("vector-valued NormalGamma (mixture precisions) is SURVEY §8 f2 (next)")
        ss_vec, cnt_vec, qname = engine.get_quadratic_form(plan, host_state, nrm)
        a0, b0 = st[gam.shape.form], st[gam.rate.form]
        ctx = plan.ctx(self)
        if "rng" not in ctx:
            ctx["rng"] = plan.rng_site()
            ctx["dg"], ctx["dg_stride"] = (None, 0)
            if debug_draws and "g" in debug_draws:
                ctx["dg"], ctx["dg_stride"] = plan.debug_tensor(debug_draws["g"], 1)
            ctx["probes"] = None
            if plan.probes is not None and plan.probes.get("enable"):
                plan.probes[self.param] = ctx["probes"] = {"a": plan.new(C), "b": plan.new(C)}
        rng, dg, dg_stride, probes = ctx["rng"], ctx["dg"], ctx["dg_stride"], ctx["probes"]
        plan.require(qname)

        def ngargs():
            return (C, a0.vec(), b0.vec(), ss_vec(), cnt_vec(), out.data, rng), dict(
                debug_g=dg, probe_a=probes["a"] if probes else None, probe_b=probes["b"] if probes else None,
                debug_sweep_stride=dg_stride)

        def launch():
            a, kw = ngargs()
            K.ng_draw(*a, **kw)

        def fop():
            a, kw = ngargs()
            return K.fop_ng_draw(*a, **kw)

        plan.emit(launch, f"ng_draw[{self.param}]", fop=fop)
        plan.wrote(self.param)

    def _compile_mixture(self, plan, host_state, gam, nrm, debug_draws):
        """The K-loop of sampler.py:281-284 over the components of a MixtureParameterMatrix precision: a*_k = a_k +
        n_k / 2, b*_k = b_k + sum_{z_i = k} (x_i - mu[z_i])^2 / 2 (parameter.py:522-538: the un-scaled precision of
        component k is the 0/1 diagonal of its allocation matches), all K Gamma draws in one launch."""
        st = plan.state
        C = st.n_chains
        mix = engine.get_mixture(plan, host_state, nrm)
        out = st[self.param]
        a0, b0 = st[gam.shape.form], st[gam.rate.form]
        for v, what in ((a0, "shape"), (b0, "rate")):
            if v.size not in (1, mix.K):
                raise engine.PlanError(f"NormalGamma: Gamma {what} of size {v.size} for {mix.K} mixture components")
        ctx = plan.ctx(self)
        if "rng" not in ctx:
            ctx["rng"] = plan.rng_site()
            ctx["dg"], ctx["dg_stride"] = (None, 0)
            if debug_draws and "g" in debug_draws:
                ctx["dg"], ctx["dg_stride"] = plan.debug_tensor(debug_draws["g"], mix.K)
            ctx["probes"] = None
            if plan.probes is not None and plan.probes.get("enable"):
                plan.probes[self.param] = ctx["probes"] = {"a": plan.new(C, mix.K), "b": plan.new(C, mix.K)}
        rng, dg, dg_stride, probes = ctx["rng"], ctx["dg"], ctx["dg_stride"], ctx["probes"]
        plan.require(mix.qname)
        stride = mix.K * 4

        def ngargs():
            return (C, a0.vec(), b0.vec(), K.vec((mix.stats[:, 0, 2:], stride)), K.vec((mix.stats, stride)), out.data,
                    rng), dict(debug_g=dg, probe_a=probes["a"] if probes else None, probe_b=probes["b"] if probes else None,
                               debug_sweep_stride=dg_stride, n_elem=mix.K, a0_len=a0.size, b0_len=b0.size, ss_stride=4,
                               cnt_stride=4)

        def launch():
            a, kw = ngargs()
            K.ng_draw(*a, **kw)

        def fop():
            a, kw = ngargs()
            return K.fop_ng_draw(*a, **kw)

        plan.emit(launch, f"ng_draw[{self.param}]", fop=fop)
        plan.wrote(self.param)


@dataclass
class MixtureAllocation(MCMCSampler):
    """Conjugate draw of the allocations of a mixture Normal: z_i ~ Cat(gam_i), gam_ik proportional to
    prob_k N(x_i; mu_k, 1/tau_k).  ref: sampler.py:292-355.  `debug_draws={"u": ...}` injects the uniforms of the
    reference's uniform.rvs(size=(n, 1))."""

    response_param: Union[str, None] = None

    def __post_init__(self):
        from openmcmc_b200.distribution.distribution import Categorical

        self.model = Model([self.model[self.param], self.model[self.response_param]])
        nrm = self.model[self.response_param]
        if not isinstance(nrm, Normal):
            raise TypeError("Mixture model currently only implemented for Normal case")
        if not isinstance(nrm.mean, MixtureParameterVector):
            raise TypeError("Mean must be of type MixtureParameterVector")
        if not isinstance(nrm.precision, MixtureParameterMatrix):
            raise TypeError("Mean must be of type MixtureParameterMatrix")
        if not isinstance(self.model[self.param], Categorical):
            raise TypeError("the allocation parameter needs a Categorical prior")

    def compile(self, plan, host_state, debug_draws=None):
        st = plan.state
        C = st.n_chains
        nrm = self.model[self.response_param]
        mix = engine.get_mixture(plan, host_state, nrm)
        prob = st[self.model[self.param].prob.form]
        if prob.cols != mix.K or prob.rows not in (1, mix.n):
            raise engine.PlanError(f"allocation prior of shape ({prob.rows},{prob.cols}) for {mix.n} responses and "
                                   f"{mix.K} components")
        ctx = plan.ctx(self)
        if "rng" not in ctx:
            ctx["rng"] = plan.rng_site()
            ctx["du"], ctx["du_stride"] = (None, 0)
            if debug_draws and "u" in debug_draws:
                ctx["du"], ctx["du_stride"] = plan.debug_tensor(debug_draws["u"], mix.n)
        rng, du, du_stride = ctx["rng"], ctx["du"], ctx["du_stride"]

        def launch():
            K.mixture_allocation(C, mix.n, mix.K, mix.x.vec(), mix.mu.vec(), mix.tau.vec(), prob.vec(), prob.rows,
                                 mix.z.data, rng, debug_u=du, debug_sweep_stride=du_stride)

        plan.emit(launch, f"mixture_allocation[{self.param}]")
        plan.wrote(self.param)
