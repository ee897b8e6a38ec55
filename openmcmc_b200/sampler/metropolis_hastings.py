"""Metropolis-Hastings samplers (host-side mirror).  ref: sampler/metropolis_hastings.py:25-373"""

from abc import abstractmethod
from dataclasses import dataclass, field
from typing import Callable

import numpy as np

from openmcmc_b200.sampler.sampler import MCMCSampler


@dataclass
class AcceptRate:
    """Acceptance-rate bookkeeping.  ref: metropolis_hastings.py:25-66 (counts are summed over chains)."""

    def __init__(self):
        self.count = {"accept": 0, "proposal": 0}

    @property
    def acceptance_rate(self) -> float:
        return self.count["accept"] / self.count["proposal"] * 100

    def get_acceptance_rate(self) -> str:
        if self.count["proposal"] == 0:
            return "No proposals"
        return f"Acceptance rate {self.acceptance_rate:.0f}%"

    def increment_accept(self):
        self.count["accept"] += 1

    def increment_proposal(self):
        self.count["proposal"] += 1


@dataclass
class MetropolisHastings(MCMCSampler):
    """ref: metropolis_hastings.py:69-173.  The accept/reject step (log U < log alpha, strict; NaN rejects) runs
    inside the proposal kernels; per-chain accept/proposal counters live on the device."""

    step: np.ndarray = field(default_factory=lambda: np.array([0.2], ndmin=2), init=True)
    accept_rate: AcceptRate = field(default_factory=lambda: AcceptRate(), init=False)

    def _rj_of(self, plan):
        """The ReversibleJump sampler whose padded state holds self.param (None when there is none)."""
        rj = plan.__dict__.get("_rj")
        if rj is None or rj.basis is None:
            return None
        names = (rj.basis.knots, rj.basis.widths, rj.matching_params["variable"])
        return rj if self.param in names else None

    def _collect_accept(self, plan):
        ctx = plan.ctx(self)
        cnt = ctx.get("counters")
        if cnt is not None:
            c = cnt.cpu().numpy()
            self.accept_rate.count["accept"] += int(c[:, 0].sum())
            self.accept_rate.count["proposal"] += int(c[:, 1].sum())
            self.accept_counts = c.copy()
            cnt.zero_()

    def _after_sample(self, plan):
        self._collect_accept(plan)

    def _mh_context(self, plan, n_steps, p_prop, debug_draws):
        """RNG site, per-chain counters and injected proposal / accept variates (shared by all MH kernels)."""
        import torch

        ctx = plan.ctx(self)
        if "rng" not in ctx:
            C = plan.state.n_chains
            ctx["rng"] = plan.rng_site()
            ctx["counters"] = torch.zeros(C, 2, dtype=torch.int64, device=plan.state.device)
            ctx["dz"], ctx["dz_stride"], ctx["du"], ctx["du_stride"] = None, 0, None, 0
            if debug_draws:
                zkey = "z" if "z" in debug_draws else ("tn_u" if "tn_u" in debug_draws else None)
                if zkey:
                    ctx["dz"], ctx["dz_stride"] = plan.debug_tensor(debug_draws[zkey], n_steps * p_prop)
                if "u" in debug_draws:
                    ctx["du"], ctx["du_stride"] = plan.debug_tensor(debug_draws["u"], n_steps)
        return ctx


@dataclass
class RandomWalk(MetropolisHastings):
    """Gaussian / truncated-Gaussian random-walk proposals, all elements at once.  ref: metropolis_hastings.py:176-269

    `state_update_function` is a Python callback over the dict state (SURVEY F10) and cannot run inside a kernel:
    giving one raises PlanError at compile time.
    """

    domain_limits: np.ndarray = None
    state_update_function: Callable = None
    rj: object = None      # extension: the ReversibleJump sampler of the model when this sampler runs without it
    _loop = 0

    def __post_init__(self):
        """ref: metropolis_hastings.py:201-210 (the full model is kept when a state_update_function is given)"""
        if self.state_update_function is None:
            self.model = self.model.conditional(self.param)
        self.step = np.array(self.step, ndmin=2, dtype=np.float64)

    def compile(self, plan, host_state, debug_draws=None):
        from openmcmc_b200 import devdist, engine
        from openmcmc_b200 import kernels as K

        rj = self._rj_of(plan)
        if rj is not None:
            return self._compile_rj_walk(plan, rj, debug_draws)
        if callable(self.state_update_function):
            raise engine.PlanError("state_update_function is a Python callback and cannot run on the device (SURVEY F10)")
        st = plan.state
        theta = st[self.param]
        p_dim, n_rep = theta.rows, theta.cols
        loop = self._loop
        if loop and self.domain_limits is None and (n_rep > 1 or p_dim > 1):
            # the reference raises here as well (SURVEY F5; metropolis_hastings.py:250,262): column mu of shape (p_dim,)
            # plus a full-shape normal (p_dim, n_rep) cannot be assigned back into one column unless both are 1
            shape = (p_dim, n_rep) if n_rep > 1 else (p_dim, p_dim)
            raise ValueError(f"could not broadcast input array from shape {shape} into shape ({p_dim},)")
        n_steps = n_rep if loop else 1
        p_prop = p_dim if loop else p_dim * n_rep
        model, _ = devdist.build_terms(plan, host_state, self.model, self.param)
        ctx = self._mh_context(plan, n_steps, p_prop, debug_draws)
        if "step" not in ctx:
            step = np.ascontiguousarray(self.step, dtype=np.float64)
            if step.shape[0] not in (1, p_dim) or step.shape[1] not in (1, n_rep):
                raise ValueError(f"step of shape {step.shape} does not match the parameter shape ({p_dim},{n_rep})")
            import torch

            ctx["step"] = torch.as_tensor(step).to(st.device)
            ctx["step_shape"] = step.shape
            ctx["limits"] = None
            if self.domain_limits is not None:
                lim = np.ascontiguousarray(np.asarray(self.domain_limits, dtype=np.float64).reshape(-1, 2))
                if lim.shape[0] != p_dim:
                    raise ValueError(f"domain_limits must have shape ({p_dim}, 2)")
                ctx["limits"] = torch.as_tensor(lim).to(st.device)
            ctx["probe"] = None
            if plan.probes is not None and plan.probes.get("enable"):
                ctx["probe"] = plan.new(st.n_chains, n_steps, 5)
                plan.probes[self.param] = {"steps": ctx["probe"]}

        def launch():
            K.random_walk(model, theta.data, p_dim, n_rep, loop, K.vec(ctx["step"]), ctx["step_shape"][0],
                          ctx["step_shape"][1], ctx["limits"], ctx["rng"], debug_z=ctx["dz"], debug_u=ctx["du"],
                          stride_z=ctx["dz_stride"], stride_u=ctx["du_stride"], counters=ctx["counters"],
                          probe=ctx["probe"])

        plan.emit(launch, f"{'random_walk_loop' if loop else 'random_walk'}[{self.param}]")
        plan.wrote(self.param)


    def extra_state_names(self):
        """State this sampler rewrites besides self.param: the basis matrix when it moves RJ knots / widths (MCMC's
        warm-up pass saves and restores it together with the sampled parameter)."""
        rj = getattr(self, "_rj_bound", None)
        return [rj.basis.matrix] if rj is not None else []

    def _compile_rj_walk(self, plan, rj, debug_draws):
        """Knots / widths of a ReversibleJump model: one truncated step per live component with the basis column
        rebuilt for the proposal (omc_rj_knot_walk).  The basis is the RJ sampler's declared GaussianKernelBasis; a
        `state_update_function` given for reference compatibility (its tests pass make_basis) is not called."""
        from openmcmc_b200 import engine
        from openmcmc_b200 import kernels as K

        if not self._loop:
            raise engine.PlanError("knots / widths of a ReversibleJump model are moved by RandomWalkLoop")
        self._rj_bound = rj
        if self.domain_limits is None:
            raise ValueError("RandomWalkLoop needs domain_limits (SURVEY F5)")
        lim = np.asarray(self.domain_limits, dtype=np.float64).reshape(-1, 2)
        step = np.asarray(self.step, dtype=np.float64)
        if lim.shape[0] != 1 or step.size != 1:
            raise engine.PlanError("RandomWalkLoop on RJ knots / widths needs one (lower, upper) pair and a scalar step")
        args = rj.setup(plan, None)
        which = 0 if self.param == rj.basis.knots else 1
        n_max = int(rj.n_max)
        import torch

        ctx = plan.ctx(self)
        if "rng" not in ctx:
            ctx["rng"] = plan.rng_site()
            ctx["counters"] = torch.zeros(plan.state.n_chains, 2, dtype=torch.int64, device=plan.state.device)
            ctx["dz"], ctx["du"], ctx["stride"] = None, None, 0
            if debug_draws:
                if "tn_u" in debug_draws:
                    ctx["dz"], ctx["stride"] = plan.debug_tensor(debug_draws["tn_u"], n_max)
                if "u" in debug_draws:
                    ctx["du"], ctx["stride"] = plan.debug_tensor(debug_draws["u"], n_max)

        def launch():
            K.rj_knot_walk(args, which, float(step.item()), lim[0, 0], lim[0, 1], debug_tn_u=ctx["dz"], debug_u=ctx["du"],
                           debug_sweep_stride=ctx["stride"], counters=ctx["counters"], rng_=ctx["rng"])

        plan.emit(launch, f"rj_knot_walk[{self.param}]")
        plan.wrote(self.param)
        plan.wrote(rj.basis.matrix)


@dataclass
class RandomWalkLoop(RandomWalk):
    """One MH step per replicate column of the (p_dim, n_rep) parameter.  ref: metropolis_hastings.py:272-289"""

    _loop = 1


@dataclass
class ManifoldMALA(MetropolisHastings):
    """Manifold MALA: N(theta + 1/2 s^2 H^-1 g, s^2 H^-1) forward and reverse.  ref: metropolis_hastings.py:292-373

    derivatives = "analytic" (default) uses closed-form gradients / Hessians of the Poisson / Gamma / Normal terms;
    "fd" evaluates the reference's central finite-difference stencil (distribution.py:124-198) in-kernel (parity mode).
    An invalid proposal (outside the support, non-PD Hessian) is rejected and flagged in the chain's status word; the
    reference raises instead (SURVEY F6).
    """

    derivatives: str = "analytic"
    rj: object = None      # extension: see RandomWalk.rj

    def _compile_rj(self, plan, rj, debug_draws):
        """Coefficients of a ReversibleJump model (variable length on the padded state): omc_rj_coef_mmala."""
        import torch

        from openmcmc_b200 import engine
        from openmcmc_b200 import kernels as K

        step = np.asarray(self.step, dtype=np.float64)
        if step.size != 1:
            raise engine.PlanError("ManifoldMALA on the device needs a scalar step")
        args = rj.setup(plan, None)
        n_max = int(rj.n_max)
        C = plan.state.n_chains
        ctx = plan.ctx(self)
        if "rng" not in ctx:
            ctx["rng"] = plan.rng_site()
            ctx["counters"] = torch.zeros(C, 2, dtype=torch.int64, device=plan.state.device)
            ctx["dz"], ctx["dz_stride"], ctx["du"], ctx["du_stride"] = None, 0, None, 0
            if debug_draws:
                if "z" in debug_draws:
                    ctx["dz"], ctx["dz_stride"] = plan.debug_tensor(debug_draws["z"], n_max)
                if "u" in debug_draws:
                    ctx["du"], ctx["du_stride"] = plan.debug_tensor(debug_draws["u"], 1)
            ctx["probe"] = None
            if plan.probes is not None and plan.probes.get("enable"):
                ctx["probe"] = plan.new(C, 6, fill=0.0)
                plan.probes[self.param] = {"step": ctx["probe"]}

        def launch():
            K.rj_coef_mmala(args, float(step.item()), debug_z=ctx["dz"], debug_u=ctx["du"], stride_z=ctx["dz_stride"],
                            stride_u=ctx["du_stride"], counters=ctx["counters"], probe=ctx["probe"], rng_=ctx["rng"])

        plan.emit(launch, f"rj_coef_mmala[{self.param}]")
        plan.wrote(self.param)

    @staticmethod
    def _wide_workspace(plan, model, n, method):
        """Above 64 parameters (omc.h, omc_mmala): an element-wise model (every term a sum over elements, analytic
        derivatives) runs up to 4096 elements; any other model runs its dense Hessian through the blocked Cholesky up to
        p = 512, with finite differences only where the reference itself is analytic (Normal, LogNormal, Normal-linear
        terms).  Returns the per-plan factor workspace the dense path needs above p = 136, or None."""
        from openmcmc_b200 import engine
        from openmcmc_b200 import kernels as K

        terms = [model.terms[i] for i in range(model.n_terms)]
        separable = method == 0 and all(
            t.kind in (K.TERM_POISSON_RATE, K.TERM_GAMMA_RESPONSE, K.TERM_UNIFORM_RESPONSE)
            or (t.kind == K.TERM_NORMAL_RESPONSE and t.mat_kind != K.MAT_DENSE) for t in terms)
        if separable:
            if n > 4096:
                raise engine.PlanError(f"ManifoldMALA on an element-wise model with n={n} > 4096 elements is not "
                                       "supported by the device path")
            return None
        if n > 512:
            raise engine.PlanError(f"ManifoldMALA with a dense Hessian and p={n} > 512 parameters is not supported by "
                                   "the device path")
        if method == 1 and any(t.kind not in (K.TERM_NORMAL_RESPONSE, K.TERM_LOGNORMAL_RESPONSE, K.TERM_NORMAL_LINEAR)
                               for t in terms):
            raise engine.PlanError(f"ManifoldMALA with derivatives='fd' and p={n} > 64 parameters needs every term "
                                   "Normal, LogNormal or Normal-linear; use derivatives='analytic'")
        ws = K.nn_dense_workspace(plan.state.n_chains, n)
        return plan.new(ws) if ws > 0 else None

    def compile(self, plan, host_state, debug_draws=None):
        from openmcmc_b200 import devdist, engine
        from openmcmc_b200 import kernels as K

        if self.derivatives not in ("analytic", "fd"):
            raise ValueError("derivatives must be 'analytic' or 'fd'")
        rj = self._rj_of(plan)
        if rj is not None:
            return self._compile_rj(plan, rj, debug_draws)
        st = plan.state
        C = st.n_chains
        theta = st[self.param]
        if theta.cols != 1:
            raise engine.PlanError("ManifoldMALA on the device needs a (p, 1) parameter")
        n = theta.rows
        step = np.asarray(self.step, dtype=np.float64)
        if step.size != 1:
            raise engine.PlanError("ManifoldMALA on the device needs a scalar step")
        method = 1 if self.derivatives == "fd" else 0
        model, _ = devdist.build_terms(plan, host_state, self.model, self.param)
        workspace = self._wide_workspace(plan, model, n, method) if n > 64 else None
        ctx = self._mh_context(plan, 1, n, debug_draws)
        if "probes" not in ctx:
            ctx["probes"] = None
            if plan.probes is not None and plan.probes.get("enable"):
                ctx["probes"] = {"mu": plan.new(C, n), "L": plan.new(C, n, n), "prop": plan.new(C, n),
                                 "scalars": plan.new(C, 6)}
                plan.probes[self.param] = ctx["probes"]
        pr = ctx["probes"] or {}

        def launch():
            K.mmala(model, theta.data, float(step.item()), method, ctx["rng"], debug_z=ctx["dz"], debug_u=ctx["du"],
                    stride_z=ctx["dz_stride"], stride_u=ctx["du_stride"], counters=ctx["counters"], status=plan.status,
                    probe_mu=pr.get("mu"), probe_L=pr.get("L"), probe_prop=pr.get("prop"),
                    probe_scalars=pr.get("scalars"), workspace=workspace)

        plan.emit(launch, f"mmala[{self.param}]")
        plan.wrote(self.param)
