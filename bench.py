#!/usr/bin/env python
"""bench.py — chain-iterations/s of the openMCMC hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload c2|c1|c3|c4a|c4b|c5|c5full]
                    [--dump-outputs DIR]

A "step" is one sweep (every sampler once) over all chains of the workload; `value` = chain-iterations/s with the
inputs resident in HBM; `e2e` = the same metric through the public API (`MCMC(...).run_mcmc()`) with HOST inputs, the
host->device upload and the device->host sample download inside the timed region.  N > 1: one process per GPU
(torchrun), chains sharded by rank (weak scaling, no data-path collective), time = max over ranks; the line also
carries a `strong` sub-record (the workload's chain count divided over the ranks).
`--impl reference` times the UNMODIFIED reference (openmcmc 1.0.7 from baseline/_ref, baseline/ref_bench.py) on the
host cores -- one `MCMC.run_mcmc()` per chain, one process per core; the numpy port (oracle/cpu_bench.py) only when
baseline/_ref is absent.

Default workload = BASELINE.json configs[1] (batched Bayesian linear regression), the configuration the metric is
quoted on that fits one GPU; its line also carries a compact `c3` sub-record (configs[2], the other configuration the
north-star target names).  The other configs are selectable for the per-config numbers in DESIGN.md / profiles/.
"""

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "chain-iterations/sec"
UNIT = "chain-iterations/s"

# cpu: bounded sample of the numpy port (oracle/cpu_bench.py); ref: bounded sample of the unmodified reference
# (baseline/ref_bench.py), both per worker process; sized for ~10-30 s of CPU work per call
WORKLOADS = {
    # BASELINE.json configs[1]: batched Bayesian linear regression (the config the metric is quoted on; fits 1 GPU)
    "c2": dict(name="batched Bayesian linear regression: 4096 chains/GPU, n=10000, p=64, NormalNormal+NormalGamma Gibbs",
               kind="regression", chains=4096, n=10000, p=64, thin=1, dominant="nn_dense_draw", flush_l2=True,
               cpu=dict(chains_per_worker=8, sweeps=100), ref=dict(chains_per_worker=1, sweeps=200),
               ref_step=dict(chains_per_worker=1, sweeps=10)),
    # BASELINE.json configs[0]: example-3 regression, single chain (latency bound)
    "c1": dict(name="examples/3_linear_regression: 1 chain, n=1000, p=3", kind="regression", chains=1, n=1000, p=3,
               thin=1, dominant="nn_dense_draw", cpu=dict(chains_per_worker=1, sweeps=4000),
               ref=dict(chains_per_worker=1, sweeps=3000), ref_step=dict(chains_per_worker=1, sweeps=200)),
    # BASELINE.json configs[2]: example-4 GMRF smoother scaled up (sparse-enabled form, SURVEY F4)
    "c3": dict(name="temporal GMRF smoother: 64 chains/GPU, n=1e6 grid points, tridiagonal NormalNormal + 2x NormalGamma",
               kind="gmrf", chains=64, n=1_000_000, p=0, thin=10, dominant="tridiag_nn_draw",
               cpu=dict(chains_per_worker=1, sweeps=3), ref=dict(chains_per_worker=1, sweeps=3),
               ref_step=dict(chains_per_worker=1, sweeps=1)),
    # BASELINE.json configs[3]: 65,536 chains x 32 params over 8 GPUs = 8192 chains per GPU
    "c4a": dict(name="ManifoldMALA, Poisson counts + Gamma prior: 8192 chains/GPU x 32 params", kind="mh", chains=8192,
                n=0, p=32, thin=1, dominant="mmala", cpu=dict(chains_per_worker=1, sweeps=30),
                ref=dict(chains_per_worker=1, sweeps=8), ref_step=dict(chains_per_worker=1, sweeps=1)),
    "c4b": dict(name="RandomWalkLoop (truncated proposals), Poisson counts + Gamma prior: 8192 chains/GPU x (1,32) params",
                kind="mh", chains=8192, n=0, p=32, thin=1, dominant="random_walk_loop",
                cpu=dict(chains_per_worker=4, sweeps=300), ref=dict(chains_per_worker=1, sweeps=300),
                ref_step=dict(chains_per_worker=1, sweeps=20)),
    # BASELINE.json configs[4]: ReversibleJump on the Gaussian-kernel basis model, 8192 chains, capacity 128 components
    "c5": dict(name="ReversibleJump birth/death, Gaussian-kernel basis model: 8192 chains/GPU, n_data=512, n_max=128, "
                    "rho=32, Normal response, matched transitions", kind="rj", chains=8192, n=512, p=128, thin=1,
               dominant="reversible_jump", cpu=dict(chains_per_worker=2, sweeps=300),
               ref=dict(chains_per_worker=1, sweeps=1000), ref_step=dict(chains_per_worker=1, sweeps=60)),
    # the same model with all four samplers of the reference's RJ model: ManifoldMALA on the coefficients, RandomWalkLoop
    # on knots and widths (basis rebuilt per proposal), ReversibleJump
    "c5full": dict(name="full RJ source model: ManifoldMALA(beta) + RandomWalkLoop(theta) + RandomWalkLoop(omega) + "
                        "ReversibleJump, 8192 chains/GPU, n_data=512, n_max=128, rho=32", kind="rj", full=True, chains=8192,
                   n=512, p=128, thin=1, dominant="reversible_jump", cpu=dict(chains_per_worker=1, sweeps=40),
                   ref=dict(chains_per_worker=1, sweeps=30), ref_step=dict(chains_per_worker=1, sweeps=3)),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--chains", type=int, default=None, help="override chains per GPU (debug only)")
    ap.add_argument("--n", type=int, default=None, help="override n (debug only)")
    ap.add_argument("--upload-blocks", type=int, default=None,
                    help="chain blocks of the e2e run (upload of block k+1 under the sweeps of block k); default: "
                         "MCMC's automatic choice, one block per 2.7 GB of per-chain host input, at most 16")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the comparison legs (sweep forms, fitted values, ESS "
                                                             "run, c3 sub-record, strong scaling)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last timed step's stored iteration of every array in "
                         "MCMC.store (rank 0's chains) as DIR/<name>.npy, float64, at most 64 MB in all (a fixed "
                         "seeded sample of the elements of an array too large for that)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the b200 implementation; --impl reference has none to dump")
    return args


def config_of(args, wl):
    """The same keys and values in both arms (the driver compares them)."""
    return {"workload": wl["name"], "chains_per_gpu": args.chains or wl["chains"], "n_obs": args.n or wl["n"],
            "p": wl["p"], "n_thin": wl["thin"], "fitted_values": False,
            "l2": "c2: the steady-state sweep touches 86 MB of its 136 MB record set (lower block triangle), which does not "
                  "clearly exceed the 126 MB L2, so a 256 MB buffer is written before EVERY timed sweep and each sweep has its "
                  "own event pair (`l2_warm` is the same run without the flushes); c3: 512 MB of y + 1 GB of scratch per "
                  "sweep, c5: 4.3 GB of basis matrices -- far larger than L2; c1/c4 working sets are L2-resident by nature of "
                  "the workload",
            "per_step": "1 sweep = every sampler once over all chains; every n_thin-th sweep also stores the samples and "
                        "log_post (no fitted values: response=None in both arms; `with_fitted_values` is the same "
                        "workload with response={'y': 'mean'})"}


# --------------------------------------------------------------------------------------------- CPU legs
def cpu_sample(key, wl, n, p, sizes, seed=0, prefer_reference=True):
    """One bounded sample of the workload on all host cores: the unmodified reference when baseline/_ref travels with
    the repo, else the numpy port.  Returns (result dict of run_parallel, kind)."""
    cores = os.cpu_count() or 1
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    try:
        import ref_bench
    except Exception:
        ref_bench = None
    if prefer_reference and ref_bench is not None and ref_bench.available():
        r = ref_bench.run_parallel(workload=key, workers=cores, n=n, p=p, seed=seed, n_thin=1, **sizes["ref"])
        return r, "reference"
    from oracle import cpu_bench

    r = cpu_bench.run_parallel(workload=key, workers=cores, n=n, p=p, seed=seed, **sizes["cpu"])
    return r, "port"


def run_reference(args, wl, key):
    """`--impl reference`: W untimed + K timed steps, each step one bounded sample on every host core."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n, p = args.n or wl["n"], wl["p"]
    sizes = {"ref": wl["ref_step"], "cpu": wl["ref_step"]}
    kind = None
    for k in range(args.warmup):
        _, kind = cpu_sample(key, wl, n, p, sizes, seed=50 + k)
    secs, its, failed, last = 0.0, 0, 0, None
    for k in range(args.steps):
        r, kind = cpu_sample(key, wl, n, p, sizes, seed=100 + k)
        secs += r["seconds"]
        its += r["cores"] * wl["ref_step"]["chains_per_worker"] * wl["ref_step"]["sweeps"]
        failed += r.get("chains_failed", 0)
        last = r
    value = its / secs
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": secs / max(args.steps, 1) * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config_of(args, wl),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": last["cores"], "kind": kind,
                         "sample": f"{args.steps} steps, each: {last['sample']}"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "chains_failed": failed,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []      # (host time, csv line)
        self.proc = None
        self.t_mark = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def mark(self):
        """Start of the timed region: the sampler itself starts before the warm-up (nvidia-smi needs a second or more
        to come up on an 8-GPU node), samples from here on are the ones reported."""
        self.t_mark = time.perf_counter()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        timed = [r for t, r in self.rows if self.t_mark is None or t >= self.t_mark]
        window = "timed region + dominant-op timing"
        if not timed:     # the timed region was shorter than one sampling period: report the warm-up samples instead
            timed, window = [r for _, r in self.rows], "warm-up + timed region (timed region shorter than one sample)"
        for r in timed:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        med = sm[len(sm) // 2] if sm else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm), "window": window}


# --------------------------------------------------------------------------------------------- workloads (B200 arm)
def build_regression(C, n, p, dev, rank, host, response=False):
    import numpy as np
    import torch
    from scipy import sparse

    from openmcmc_b200.distribution.distribution import Gamma
    from openmcmc_b200.distribution.location_scale import Normal
    from openmcmc_b200.model import Model
    from openmcmc_b200.parameter import LinearCombination, ScaledMatrix
    from openmcmc_b200.sampler.sampler import NormalGamma, NormalNormal

    # synthetic data generated on the device (SURVEY §8d: X = [1, N(0,1)...], y = X beta* + 0.1 eps), seed = rank
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    X = torch.randn(C, n, p, dtype=torch.float64, device=dev, generator=gen)
    X[:, :, 0] = 1.0
    beta_true = torch.randn(C, p, 1, dtype=torch.float64, device=dev, generator=gen)
    y = torch.bmm(X, beta_true) + 0.1 * torch.randn(C, n, 1, dtype=torch.float64, device=dev, generator=gen)
    if host:
        X, y = _pinned(X), _pinned(y)
    mdl = Model([
        Normal("y", mean=LinearCombination(form={"beta": "X"}), precision=ScaledMatrix(matrix="P_tau", scalar="tau")),
        Normal("beta", mean="mu", precision=ScaledMatrix(matrix="P_lambda", scalar="lambda")),
        Gamma("tau", shape="a_tau", rate="b_tau"),
        Gamma("lambda", shape="a_lambda", rate="b_lambda")], response={"y": "mean"} if response else None)
    samplers = [NormalNormal("beta", mdl), NormalGamma("tau", mdl), NormalGamma("lambda", mdl)]
    state = {"y": y, "X": X, "beta": np.zeros((p, 1)), "P_tau": sparse.identity(n, format="csc"), "tau": 1.0,
             "P_lambda": sparse.identity(p, format="csc"), "mu": np.zeros((p, 1)), "lambda": 0.01,
             "a_tau": 1e-3, "b_tau": 1e-3, "a_lambda": 1e-3, "b_lambda": 1e-3}
    return mdl, samplers, state


def build_gmrf(C, n, p, dev, rank, host):
    """SURVEY §8d C3: regular grid s_i = i*(60/99), P = precision_irregular(s), P[0,0] += 1e-3,
    y = sin(s/20) + 2 cos(s/12) + 2 + eps; lambda0 = 100, a_lam = 10, b_lam = 1, tau0 = 1, a_tau = b_tau = 1."""
    import numpy as np
    import torch
    from scipy import sparse

    from openmcmc_b200.distribution.distribution import Gamma
    from openmcmc_b200.distribution.location_scale import Normal
    from openmcmc_b200.model import Model
    from openmcmc_b200.parameter import LinearCombination, ScaledMatrix
    from openmcmc_b200.sampler.sampler import NormalGamma, NormalNormal

    s = np.arange(n) * (60.0 / 99.0)
    dr = 1.0 / np.diff(s)
    pd = np.append(np.append(dr[0], dr[:-1] + dr[1:]), dr[-1])
    pd[0] += 1e-3
    P = sparse.diags([-dr, pd, -dr], offsets=[-1, 0, 1], format="csc")
    gen = torch.Generator(device=dev)
    gen.manual_seed(4321 + rank)
    truth = torch.as_tensor(np.sin(s / 20) + 2 * np.cos(s / 12) + 2).to(dev)
    y = truth.reshape(1, n, 1) + torch.randn(C, n, 1, dtype=torch.float64, device=dev, generator=gen)
    if host:
        y = _pinned(y)
    mdl = Model([Normal("y", mean=LinearCombination(form={"b": "I"}), precision=ScaledMatrix(matrix="P_tau", scalar="tau")),
                 Normal("b", mean="mu", precision=ScaledMatrix(matrix="P_lambda", scalar="lambda")),
                 Gamma("lambda", shape="a_lam", rate="b_lam"),
                 Gamma("tau", shape="a_tau", rate="b_tau")])
    samplers = [NormalNormal("b", mdl), NormalGamma("lambda", mdl), NormalGamma("tau", mdl)]
    state = {"y": y, "b": y, "mu": np.zeros(n), "lambda": 100, "P_lambda": P, "a_lam": 10, "b_lam": 1, "tau": 1,
             "P_tau": sparse.identity(n, format="csc"), "I": sparse.identity(n, format="csc"), "a_tau": 1, "b_tau": 1}
    return mdl, samplers, state


def build_mh(C, n, p, dev, rank, host, loop):
    """SURVEY §8d C4: y_j ~ Poisson(lambda*_j), lambda* ~ Gamma(5,1), prior Gamma(2, 0.5); step 0.5."""
    import numpy as np
    import torch

    from openmcmc_b200.distribution.distribution import Gamma, Poisson
    from openmcmc_b200.model import Model
    from openmcmc_b200.sampler.metropolis_hastings import ManifoldMALA, RandomWalkLoop

    rng = np.random.default_rng(99 + rank)
    shape = (C, 1, p) if loop else (C, p, 1)
    y = rng.poisson(rng.gamma(5.0, 1.0, size=shape)).astype(np.float64)
    yt = torch.as_tensor(y)
    yt = yt.pin_memory() if host else yt.to(dev)
    mdl = Model([Poisson("y", rate="lam"), Gamma("lam", shape="a", rate="b")])
    if loop:
        smp = RandomWalkLoop("lam", mdl, step=np.array([[0.5]]), domain_limits=np.array([[0.0, np.inf]]),
                             max_variable_size=(1, p))
    else:
        smp = ManifoldMALA("lam", mdl, step=np.array([[0.5]]))
    state = {"y": yt, "lam": torch.as_tensor(y + 1.0), "a": np.array([[2.0]]), "b": np.array([[0.5]])}
    return mdl, [smp], state


def build_rj(C, n_data, n_max, dev, rank, host, full=False):
    """SURVEY §8d C5: the reference RJ test model scaled — n_data points on [-10, 10], capacity n_max, rho = n_max / 4,
    Gaussian-kernel basis, truncated matching [-10, 10] with scale 1; every chain has its own response."""
    import numpy as np
    import torch
    from scipy import sparse

    from openmcmc_b200.distribution.distribution import Gamma, Poisson, Uniform
    from openmcmc_b200.distribution.location_scale import Normal
    from openmcmc_b200.model import Model
    from openmcmc_b200.parameter import LinearCombination, MixtureParameterMatrix, MixtureParameterVector, ScaledMatrix
    from openmcmc_b200.sampler.reversible_jump import GaussianKernelBasis, ReversibleJump

    rng = np.random.default_rng(77 + rank)
    rho = n_max / 4.0
    k0 = int(rho)
    X = np.sort(rng.uniform(-10, 10, n_data))
    theta = rng.uniform(-10, 10, (C, 1, k0))
    omega = rng.uniform(0.8, 1.6, (C, 1, k0))
    beta = rng.standard_normal((C, k0, 1))
    z = (X.reshape(1, -1, 1) - theta) / omega
    Bt = np.exp(-0.5 * z * z) / (np.sqrt(2 * np.pi) * omega)                # [C, n_data, k0]
    y = Bt @ beta + 0.1 * rng.standard_normal((C, n_data, 1))
    yt = torch.as_tensor(y)
    yt = yt.pin_memory() if host else yt.to(dev)
    mdl = Model([Normal("y", mean=LinearCombination(form={"beta": "B"}), precision=ScaledMatrix(matrix="P", scalar="tau_y")),
                 Normal("beta", mean=MixtureParameterVector(param="mu_beta", allocation="alloc_beta"),
                        precision=MixtureParameterMatrix(param="tau_beta", allocation="alloc_beta")),
                 Poisson("n_basis", rate="rho"),
                 Uniform("theta", domain_response_lower=np.array([[-10.0]]), domain_response_upper=np.array([[10.0]])),
                 Gamma("omega", shape="a_omega", rate="b_omega")])
    smp = ReversibleJump(param="n_basis", model=mdl, associated_params=["theta", "omega"], n_max=n_max,
                         matching_params={"variable": "beta", "matrix": "B", "scale": 1.0, "limits": [-10.0, 10.0]},
                         basis=GaussianKernelBasis(matrix="B", locations="X", knots="theta", widths="omega"))
    state = {"y": yt, "beta": beta, "tau_y": 100.0, "P": sparse.eye(n_data), "B": np.zeros((n_data, k0)), "n_basis": k0,
             "X": X.reshape(-1, 1), "theta": theta, "omega": omega, "mu_beta": np.zeros((1, 1)),
             "tau_beta": 0.25 * np.ones((1, 1)), "rho": rho, "alloc_beta": np.zeros((k0, 1)),
             "a_omega": 3.0 * np.ones((1, 1)), "b_omega": 2.0 * np.ones((1, 1))}
    if full:
        from openmcmc_b200.sampler.metropolis_hastings import ManifoldMALA, RandomWalkLoop

        samplers = [ManifoldMALA(param="beta", model=mdl, step=np.array(0.8), max_variable_size=n_max),
                    RandomWalkLoop(param="theta", model=mdl, step=np.array(0.3), max_variable_size=n_max,
                                   domain_limits=np.array([-10.0, 10.0], ndmin=2)),
                    RandomWalkLoop(param="omega", model=mdl, step=np.array(0.1), max_variable_size=n_max,
                                   domain_limits=np.array([0.5, 2.0], ndmin=2)),
                    smp]
        return mdl, samplers, state
    return mdl, [smp], state


def _pinned(t):
    import torch

    h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    h.copy_(t)
    return h


def build(wl, C, n, dev, rank, host=False, response=False):
    if wl["kind"] == "regression":
        return build_regression(C, n, wl["p"], dev, rank, host, response)
    if wl["kind"] == "gmrf":
        return build_gmrf(C, n, wl["p"], dev, rank, host)
    if wl["kind"] == "rj":
        return build_rj(C, n, wl["p"], dev, rank, host, full=wl.get("full", False))
    return build_mh(C, n, wl["p"], dev, rank, host, loop=wl["dominant"] == "random_walk_loop")


def numa_interleave(enable: bool):
    """Memory policy of the calling thread for the pinned e2e inputs.  With several ranks per node every rank's pinned
    copy landing on the NUMA node all GPUs report as local made the upload the limiter of the round-1 scaling run
    (8 ranks x 21 GB from one node's DRAM: 18 GB/s per rank against 46-51 GB/s alone); interleaving the pages over all
    nodes spreads that load.  Returns a description for the JSON line."""
    import ctypes
    import glob

    nodes = sorted(int(os.path.basename(q)[4:]) for q in glob.glob("/sys/devices/system/node/node[0-9]*"))
    if len(nodes) < 2:
        return "default (single NUMA node)"
    libc = ctypes.CDLL("libc.so.6", use_errno=True)
    if not enable:
        libc.syscall(238, 0, None, 0)              # set_mempolicy(MPOL_DEFAULT)
        return "default"
    mask = ctypes.c_ulong(sum(1 << nd for nd in nodes))
    rc = libc.syscall(238, 3, ctypes.byref(mask), 64)   # set_mempolicy(MPOL_INTERLEAVE, all nodes)
    return f"interleave over nodes {nodes}" + ("" if rc == 0 else f" (set_mempolicy failed rc={rc}: default)")


def roofline_of(wl, C, n, p, op_ms, step_ms, peaks, fp64_peak, syrk_ms=None, key=None):
    """Algorithmic work of the dominant op per launch (DESIGN.md §3) over its measured duration."""
    hbm_peak, hbm_src = peaks
    sec = op_ms * 1e-3
    traffic, traffic_src = None, None
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", f"{key}_traffic.json")))
        traffic, traffic_src = t["dram_bytes_per_launch"], "static: " + t["source"]
    except Exception:
        pass
    common = {"peak": hbm_peak, "unit": "GB/s", "peak_source": hbm_src, "traffic": traffic,
              "traffic_source": traffic_src, "kernel_ms": op_ms, "share_of_step": op_ms / step_ms}
    if wl["kind"] == "regression":
        # per sweep and chain the draw needs the record G | g | rss | cnt -- G symmetric: p (p + 1) / 2 unique entries (the
        # kernel reads the lower block triangle, and G a second time for d'G d from L2) -- and the centre (8 (2p + 2)),
        # and writes beta (8 p) and rss: no pass over X (DESIGN.md §3.1)
        byts = C * 8 * (p * (p + 1) // 2 + p + 2 + 2 * p + 2 + p + 1)
        flops = C * (p ** 3 / 3.0 + 2.0 * p * p + 2.0 * p * p + 2.0 * p * p)   # Cholesky, 3 triangular solves, d'G d
        roof = {"bound": "hbm", "kernel": "nn draw kernel (omc_nn_dense_draw: Q = lam P0 + tau G, Cholesky, posterior "
                                          "mean, draw, re-centred rss): the whole data-dependent work of a sweep",
                "achieved": byts / sec / 1e9, "frac": byts / sec / 1e9 / hbm_peak, **common,
                "fp64": {"achieved_tflops": flops / sec / 1e12, "peak_tflops": fp64_peak,
                         "frac": flops / sec / 1e12 / fp64_peak if fp64_peak else None,
                         "flops_per_chain": flops / C,
                         "peak_source": "cuBLAS DGEMM fp64 6144^3 measured in this run"}}
        # SURVEY §8d quotes C2 on the REFERENCE algorithm's traffic -- one pass over (X, y) per chain-iteration,
        # 8 n (p + 1) bytes.  Against that figure the sweep sits above the HBM roofline because it no longer reads X
        # (re-centred statistics); `frac` above is the kernel's own bytes, this one is the contract's literal figure.
        sv = C * 8.0 * n * (p + 1)
        roof["survey_8d"] = {"bytes_per_chain_iteration": 8.0 * n * (p + 1), "achieved": sv / sec / 1e9,
                             "frac": sv / sec / 1e9 / hbm_peak, "unit": "GB/s",
                             "note": "reference-algorithm bytes (one pass over X, y per chain-iteration) / the draw "
                                     "kernel's duration: > 1 because X left the steady-state sweep"}
        if syrk_ms:
            fl = C * (n * p * (p + 1) + 4 * n * p)   # SYRK + X'y + residual per chain (SURVEY §8d)
            tf = fl / (syrk_ms * 1e-3) / 1e12
            roof["prologue_syrk"] = {
                "bound": "tensor", "kernel": "reg_pass_kernel (FP64 DMMA SYRK + X'y + rss), once per run (prologue)",
                "achieved": tf, "peak": fp64_peak, "unit": "TFLOP/s", "frac": tf / fp64_peak if fp64_peak else None,
                "peak_source": "cuBLAS DGEMM fp64 6144^3 measured in this run (MEASURED_PEAKS.json has no fp64 figure)",
                "kernel_ms": syrk_ms, "hbm_gbs": C * 8.0 * n * (p + 1) / (syrk_ms * 1e-3) / 1e9}
        return roof
    if wl["kind"] == "gmrf":
        byts = C * 32 * n                                 # read y, P diag + off, write b (SURVEY §8d)
        return {"bound": "hbm", "kernel": "omc_tridiag_nn_draw (tg_aggregate_kernel + tg_tilescan_kernel + tg_solve_kernel)",
                "achieved": byts / sec / 1e9, "frac": byts / sec / 1e9 / hbm_peak, **common}
    if wl["kind"] == "rj":
        k = p / 4.0                                       # expected live components (rho = n_max / 4)
        byts = C * 2 * 8 * n * k                          # two passes over the live basis columns (SURVEY §8d: 8 n_data k)
        flops = C * (2 * n * k * k + 4.0 / 3.0 * k ** 3)
        return {"bound": "hbm", "kernel": "rj_kernel (Gram + in-place inverse + LU per chain; latency / FP64-ALU bound)",
                "achieved": byts / sec / 1e9, "frac": byts / sec / 1e9 / hbm_peak, **common,
                "fp64": {"achieved_tflops": flops / sec / 1e12, "flops_per_chain_step": flops / C}}
    byts = C * 32 * p                                     # read theta, y; write theta, sample (SURVEY §8d)
    return {"bound": "hbm", "kernel": f"{wl['dominant']}_kernel (latency / FP64-ALU bound: 1 KB per chain-iteration)",
            "achieved": byts / sec / 1e9, "frac": byts / sec / 1e9 / hbm_peak, **common}


class Ctx:
    """Process-wide pieces of one bench run."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist

        self.args = args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        from openmcmc_b200 import kernels as K

        K.init_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.torch, self.dist, self.K = torch, dist, K

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())


L2_FLUSH_BYTES = 256 << 20


def timed_sweeps(ctx, M, steps, warmup, thin, clocks=None, flush_l2=False):
    """W untimed + exactly K timed sweeps replayed from the captured graphs (every thin-th followed by the store graph),
    CUDA events on the engine's stream, barrier + synchronize on both sides, max over ranks.  Returns ms.
    flush_l2: a 256 MB buffer is written before EVERY timed sweep and every sweep is bracketed by its own pair of events
    (the flushes are outside the brackets); the K per-sweep times are summed.  For workloads whose per-sweep working set
    does not clearly exceed the 126 MB L2 (C2 after the re-centring: the draw touches 86 MB of records per sweep)."""
    torch = ctx.torch
    n_iter = max(steps // thin, 1)
    M.run_device(n_burn=warmup, n_iter=0, n_thin=1)
    ctx.barrier()
    if clocks is not None:
        clocks.mark()
    if flush_l2 and thin == 1:
        flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=ctx.dev)
        pairs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for k, (a0, a1) in enumerate(pairs):
            with torch.cuda.stream(M.stream):
                flush.fill_(k & 255)
                a0.record()
            M.run_device(n_burn=0, n_iter=1, n_thin=1, restart_store=(k == 0))
            with torch.cuda.stream(M.stream):
                a1.record()
        ctx.barrier()
        return ctx.max_over_ranks(sum(a0.elapsed_time(a1) for a0, a1 in pairs))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(M.stream):
        e0.record()
    M.run_device(n_burn=steps % thin if steps >= thin else 0, n_iter=n_iter, n_thin=thin)
    with torch.cuda.stream(M.stream):
        e1.record()
    ctx.barrier()
    return ctx.max_over_ranks(e0.elapsed_time(e1))


def time_op(ctx, M, fn, reps=10, flush_l2=False):
    """One launch closure of the plan, captured and replayed alone on the engine's stream; events on that stream.
    flush_l2: a 256 MB buffer is written before every launch and every launch has its own event pair."""
    torch, K = ctx.torch, ctx.K
    with torch.cuda.stream(M.stream):
        g = K.Graph.capture(fn)
        g.launch(1)
        if flush_l2:
            flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=ctx.dev)
            pairs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
            for k, (a0, a1) in enumerate(pairs):
                flush.fill_(k & 255)
                a0.record()
                g.launch(1)
                a1.record()
        else:
            k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            k0.record()
            g.launch(reps)
            k1.record()
    ctx.barrier()
    if flush_l2:
        return sum(a0.elapsed_time(a1) for a0, a1 in pairs) / reps
    return k0.elapsed_time(k1) / reps


def value_leg(ctx, wl, key, C, n, steps, warmup, thin, clocks=None, chain_offset=None, response=False, stream=False,
              flush_l2=None):
    """Device-resident run of one workload: returns (M, ms over the K sweeps, state bits needed later)."""
    from openmcmc_b200.mcmc import MCMC

    mdl, samplers, state = build(wl, C, n, ctx.dev, ctx.rank, response=response)
    n_iter = max(steps // thin, 1)
    M = MCMC(state, samplers, model=mdl, n_burn=0, n_iter=n_iter, n_thin=thin, n_chains=C, seed=7, device=ctx.local,
             chain_offset=ctx.rank * C if chain_offset is None else chain_offset, stream_store=stream)
    M.prepare()
    flush = bool(wl.get("flush_l2", False)) and not response if flush_l2 is None else flush_l2
    ms = timed_sweeps(ctx, M, steps, warmup, thin, clocks, flush_l2=flush)
    return M, ms, (mdl, samplers, state)


def e2e_leg(ctx, wl, key, C, n, p, steps, thin, upload_blocks):
    """Public API with HOST (pinned) inputs: upload + plan + capture + K sweeps + download of every stored sample."""
    import contextlib
    import io

    from openmcmc_b200.mcmc import MCMC

    torch = ctx.torch
    Ce, note = C, ""
    per_chain_host = 8.0 * n * (p + 1) if wl["kind"] == "regression" else 8.0 * n * 2 if wl["kind"] == "gmrf" else 0.0
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(ctx.world)))
    try:
        import psutil

        avail = psutil.virtual_memory().available
        budget = 0.6 * avail / max(local_world, 1)
        if per_chain_host * C > budget:
            Ce = max(64, int(budget / per_chain_host) // 64 * 64)
            note = (f" [e2e on {Ce} of {C} chains per GPU: {local_world} ranks x {per_chain_host * C / 1e9:.1f} GB of "
                    f"pinned host input exceed 60% of the node's {avail / 1e9:.0f} GB of free host memory]")
    except Exception:
        pass
    policy = numa_interleave(local_world > 2)
    mdl, samplers2, hstate = build(wl, Ce, n, ctx.dev, ctx.rank, host=True)
    numa_interleave(False)
    n_iter = max(steps // thin, 1)

    mem_before = None
    prep = os.environ.get("OMC_BENCH_E2E_PREP", "")      # tuning aid: state of the caching allocator in front of the leg
    if prep:
        import gc

        gc.collect()
        st0 = torch.cuda.memory_stats()
        mem_before = {"prep": prep, "reserved_gb": st0["reserved_bytes.all.current"] / 1e9,
                      "allocated_gb": st0["allocated_bytes.all.current"] / 1e9,
                      "inactive_split_gb": st0["inactive_split_bytes.all.current"] / 1e9}
        if prep in ("empty", "warm"):
            torch.cuda.empty_cache()
        if prep == "warm":
            x = torch.empty(int(per_chain_host * Ce * 1.1), dtype=torch.uint8, device=ctx.dev)
            del x
        sys.stderr.write(f"e2e allocator state: {mem_before}\n")

    def run(blocks, first=True):
        if first:
            ctx.barrier()
        else:               # a retry on one rank must not wait on a collective the other ranks have passed
            torch.cuda.synchronize()
        t_start = time.perf_counter()
        r = MCMC(hstate, samplers2, model=mdl, n_burn=steps % thin if steps >= thin else 0, n_iter=n_iter,
                 n_thin=thin, n_chains=Ce, seed=7, device=ctx.local, chain_offset=ctx.rank * C, upload_blocks=blocks)
        prof = None
        if os.environ.get("OMC_BENCH_PROFILE"):      # host-side profile of the e2e leg (tuning aid): top of cProfile -> stderr
            import cProfile

            prof = cProfile.Profile()
            prof.enable()
        with contextlib.redirect_stdout(io.StringIO()):
            r.run_mcmc()
        if prof is not None:
            import pstats

            prof.disable()
            pstats.Stats(prof, stream=sys.stderr).sort_stats("cumulative").print_stats(40)
        return r, t_start

    try:
        M2, t0 = run(upload_blocks)
    except Exception as exc:   # never lose the whole line to the e2e leg: one more try as a single block, and say so
        note += f" [first e2e attempt failed ({type(exc).__name__}: {str(exc)[:120]}); re-run with upload_blocks=1]"
        M2, t0 = run(1, first=False)
    torch.cuda.synchronize()
    dt = ctx.max_over_ranks(time.perf_counter() - t0)
    out = {"value": Ce * ctx.world * steps / dt, "unit": UNIT, "chains_per_gpu": Ce,
           "upload_blocks": M2.timing.get("upload_blocks", 1), "streamed_store": bool(getattr(M2, "_streamed", False)),
           "h2d_bytes_per_step": M2.timing["h2d_bytes"] / steps, "d2h_bytes_per_step": M2.timing["d2h_bytes"] / steps,
           "seconds": dt, "pinned_policy": policy,
           "phases_s": {k: round(M2.timing[k], 4) for k in ("prepare_s", "sweeps_s", "collect_s") if k in M2.timing},
           "blocks": M2.timing.get("blocks"),
           "note": "MCMC(...).run_mcmc() with pinned host inputs: upload + plan compile + graph capture + "
                   f"{steps} sweeps + download of all stored samples; upload_blocks > 1: the chains run as chain "
                   "blocks, block k+1 uploading while block k sweeps; streamed_store: the stored iterations leave "
                   "the device during the sweeps (device ring -> pinned staging -> host)" + note}
    floor = M2.timing["h2d_bytes"] / 55e9 + (M2.timing["d2h_bytes"] / 55e9 if not out["streamed_store"] else 0.0)
    out["limiter"] = (f"PCIe: {M2.timing['h2d_bytes'] / 1e9:.2f} GB up + {M2.timing['d2h_bytes'] / 1e9:.2f} GB down = "
                      f"{floor:.3f} s at 55 GB/s of the {dt:.3f} s")
    del M2, hstate
    return out


DUMP_BYTES = 60 * 10 ** 6      # under 64 MB with the .npy headers


def dump_outputs(out_dir, store):
    """What a caller of the timed run receives for its last step -- the last stored iteration of every array of
    `MCMC.store` -- as out_dir/<name>.npy in float64, so that two builds can be compared output for output.  Small
    arrays are written whole; an array larger than its share of DUMP_BYTES is cut to a sample of its flat elements
    drawn with a fixed seed (sorted indices), the same for the same shapes."""
    import numpy as np

    last = {}
    for name, arr in store.items():
        a = np.asarray(arr, dtype=np.float64)
        last[name] = a[-1] if name == "log_post" else a[..., -1]    # log_post is [n_iter, C]; the rest end in n_iter
    os.makedirs(out_dir, exist_ok=True)
    budget, left = DUMP_BYTES, len(last)
    for name, a in sorted(last.items(), key=lambda kv: kv[1].nbytes):
        share = budget // left
        if a.nbytes > share:
            a = a.ravel()[np.sort(np.random.default_rng(0).choice(a.size, share // 8, replace=False))]
        budget, left = budget - a.nbytes, left - 1
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


def fp64_dgemm_peak(ctx):
    torch = ctx.torch
    a = torch.randn(6144, 6144, dtype=torch.float64, device=ctx.dev)
    b = torch.randn(6144, 6144, dtype=torch.float64, device=ctx.dev)
    best = 0.0
    for _ in range(4):
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        _ = a @ b
        g1.record()
        torch.cuda.synchronize()
        best = max(best, 2 * 6144 ** 3 / (g0.elapsed_time(g1) * 1e-3) / 1e12)
    return best


def hbm_peak():
    try:
        return (float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]),
                "MEASURED_PEAKS.json hbm_gbs (of measured)")
    except Exception:
        return (6650.0, "fallback 6.65 TB/s (of fallback)")


def ess_record(ctx, M, wl, n, ms, note_extra=""):
    """Per-chain ESS of the stored draws (device kernel), all-gather of the per-chain records over the process group
    (NCCL over NVLink when N > 1), split-R-hat / ESS on every rank (SURVEY §8e)."""
    from openmcmc_b200 import diagnostics as G

    torch = ctx.torch
    strides = {"b": max(1, n // 64)} if wl["kind"] == "gmrf" else None
    d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    d0.record()
    summ = G.summarize(M, elem_stride=strides)
    d1.record()
    torch.cuda.synchronize()
    ess_total = float(G.min_ess_per_chain(summ, all_ranks=True).sum().item())
    rhat_max = max(float(torch.nan_to_num(v["rhat"], nan=1.0).max().item()) for v in summ.values())
    bulk = None
    try:   # SURVEY §8d's estimator: bulk-ESS = ESS of the rank-normalised draws of every chain (Vehtari et al. 2021)
        sb = G.summarize(M, elem_stride=strides, rank_normalized="chain")
        bulk_total = float(G.min_ess_per_chain(sb, all_ranks=True).sum().item())
        bulk = {"value": bulk_total / (ms * 1e-3), "unit": "ESS/s", "ess_total": bulk_total}
    except Exception as exc:
        bulk = {"error": f"{type(exc).__name__}: {str(exc)[:160]}"}
    return {"value": ess_total / (ms * 1e-3), "unit": "ESS/s", "n_stored": int(M.plan.iter_counter.item()),
            "ess_total": ess_total, "bulk": bulk, "rhat_max": rhat_max, "params": sorted(summ), "diag_ms": d0.elapsed_time(d1),
            "gathered_chains": int(next(iter(summ.values()))["n_chains_total"]),
            "note": "sum over all chains of the minimum-over-parameters ESS of the stored draws, divided by the seconds "
                    "of the sweeps that produced them; per-chain records all-gathered over the process group; rhat_max "
                    "is taken ACROSS chains and is only meaningful when chains share their data (the c2/c4 workloads "
                    "give every chain its own synthetic data set, so it is large by construction)" + note_extra}


def c3_subrecord(ctx, args, peaks):
    """BASELINE configs[2] next to the default line: value, roofline of the tridiagonal draw, e2e (streamed store)."""
    wl = WORKLOADS["c3"]
    C, n, thin = wl["chains"], wl["n"], wl["thin"]
    steps = max(thin, min(args.steps, 40) // thin * thin)
    M, ms, _ = value_leg(ctx, wl, "c3", C, n, steps, min(args.warmup, 5), thin)
    op = next(fn for label, fn in M._ops["sweep"] if label.startswith(wl["dominant"]))
    op_ms = time_op(ctx, M, op)
    launches = M.launches_of(steps % thin if steps >= thin else 0, max(steps // thin, 1), thin)
    rec = {"workload": wl["name"], "value": C * ctx.world * steps / (ms * 1e-3), "unit": UNIT, "steps": steps,
           "ms_per_step": ms / steps, "n_thin": thin, "gpu_launches": launches,
           "roofline": roofline_of(wl, C, n, 0, op_ms, ms / steps, peaks, None, key="c3")} if ctx.rank == 0 else {}
    del M, op
    if not args.no_e2e:
        e2e = e2e_leg(ctx, wl, "c3", C, n, 0, steps, thin, None)
        if ctx.rank == 0:
            rec["e2e"] = e2e
    return rec


def run_b200(args, wl, key):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    C, n, p, thin = args.chains or wl["chains"], args.n or wl["n"], wl["p"], wl["thin"]
    thin = max(1, min(thin, args.steps))
    # CPU baseline first (before CUDA is initialised in this process), rank 0 at N=1 only
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu:
        r, kind = cpu_sample(key, wl, n, p, wl)
        cpu_baseline = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": kind, "sample": r["sample"]}
    ctx = Ctx(args)
    torch, K = ctx.torch, ctx.K
    from openmcmc_b200 import engine
    from openmcmc_b200.mcmc import MCMC

    clocks = ClockSampler(ctx.local)
    clocks.start()
    M, ms_max, (mdl, samplers, state) = value_leg(ctx, wl, key, C, n, args.steps, args.warmup, thin, clocks)
    n_iter = max(args.steps // thin, 1)
    gpu_launches = M.launches_of(args.steps % thin if args.steps >= thin else 0, n_iter, thin)
    # dominant op alone: the very launch closure of the sweep plan
    op = next(fn for label, fn in M._ops["sweep"] if label.startswith(wl["dominant"]))
    op_ms = time_op(ctx, M, op, flush_l2=bool(wl.get("flush_l2", False)))
    syrk_ms = None
    if wl["kind"] == "regression":   # the data-only SYRK pass of the prologue, timed the same way (it runs once per run)
        op2 = next((fn for label, fn in M._ops["prologue"] if label.startswith("reg_pass")), None)
        if op2 is not None:
            syrk_ms = time_op(ctx, M, op2)
        del op2
    clk = clocks.stop()
    ess = ess_record(ctx, M, wl, n, ms_max)
    M.collect()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, M.store)
    status_bad = int(((M.status & 3) != 0).sum())
    accept = {s.param: s.accept_rate.get_acceptance_rate() for s in samplers if hasattr(s, "accept_rate")}
    value = C * world * args.steps / (ms_max * 1e-3)
    l2_warm = None
    if wl.get("flush_l2", False):    # the same K sweeps in ONE bracket without the flushes (what round 1 and 2 quoted before)
        msw = timed_sweeps(ctx, M, args.steps, args.warmup, thin)
        l2_warm = {"value": C * world * args.steps / (msw * 1e-3), "unit": UNIT, "ms_per_step": msw / args.steps,
                   "dominant_kernel_ms": time_op(ctx, M, op),
                   "note": "no L2 flush between the sweeps: the 86 MB the draw touches per sweep partly stay in the 126 MB L2"}
    del M, op
    peaks = hbm_peak()
    fp64_peak = fp64_dgemm_peak(ctx) if wl["kind"] == "regression" else None
    extras = {}
    if l2_warm is not None:
        extras["l2_warm"] = l2_warm
    if wl["kind"] == "regression" and not args.no_extras:
        # ---- the other forms of the same sweep, on the same resident inputs
        forms = {}
        for label, flags, why in (
                ("explicit_residual_every_sweep", dict(RECENTER=False),
                 "rss from one residual-only stream over X per sweep (omc_reg_rss, HBM-bound): the round-1 plan"),
                ("syrk_every_sweep", dict(RECENTER=False, CACHE_DATA_ONLY=False),
                 "G = X'X, g = X'y and rss recomputed by the fused DMMA pass in EVERY sweep, as the reference "
                 "recomputes A'QA in every NormalNormal.sample (sampler.py:180-186)")):
            saved = {k: getattr(engine, k) for k in flags}
            for k, v in flags.items():
                setattr(engine, k, v)
            try:
                M3 = MCMC(state, samplers, model=mdl, n_burn=0, n_iter=n_iter, n_thin=thin, n_chains=C, seed=7,
                          device=ctx.local, chain_offset=rank * C, stream_store=False)
                M3.prepare()
            finally:
                for k, v in saved.items():
                    setattr(engine, k, v)
            ms3 = timed_sweeps(ctx, M3, args.steps, args.warmup, thin)
            forms[label] = {"value": C * world * args.steps / (ms3 * 1e-3), "unit": UNIT, "ms_per_step": ms3 / args.steps,
                            "note": why}
            del M3
        extras["sweep_forms"] = forms
        extras["syrk_every_sweep"] = forms["syrk_every_sweep"]
        # ---- the same workload with the reference's per-iteration fitted values (model.response = {"y": "mean"},
        #      mcmc.py:109-111): every stored iteration streams X once for X beta and writes n values per chain
        del state, mdl, samplers
        Mf, msf, _ = value_leg(ctx, wl, key, C, n, min(args.steps, 20), min(args.warmup, 3), thin, response=True)
        kf = min(args.steps, 20)
        extras["with_fitted_values"] = {
            "value": C * world * kf / (msf * 1e-3), "unit": UNIT, "steps": kf, "ms_per_step": msf / kf,
            "hbm_gbs": C * 8.0 * n * (p + 2) * kf / (msf * 1e-3) / 1e9,
            "note": "response={'y': 'mean'}: X beta per stored iteration = one read of X (8 n p) and a write of n "
                    "values per chain; HBM-bound like the round-1 residual pass"}
        del Mf, _
        # ---- ESS over >= 1000 stored draws (the 60 draws of the timed region say little about ESS)
        k_ess = 1000
        Me, mse, _ = value_leg(ctx, wl, key, C, n, k_ess, 20, thin)
        extras["ess_long"] = ess_record(ctx, Me, wl, n, mse, note_extra=f"; separate run of {k_ess} stored sweeps after 20 burn-in sweeps")
        extras["ess_long"]["ms_per_step"] = mse / k_ess
        del Me, _
    else:
        del state, mdl, samplers
    # ---- e2e: public API with HOST (pinned) inputs, upload + K sweeps + sample download inside the timed region
    import gc

    gc.collect()          # the earlier legs' device inputs (21 GB each at C2) are released before the end-to-end leg
    e2e = None if args.no_e2e else e2e_leg(ctx, wl, key, C, n, p, args.steps, thin, args.upload_blocks)
    if key == "c2" and not args.no_extras:
        try:
            extras["c3"] = c3_subrecord(ctx, args, peaks)
        except Exception as exc:
            extras["c3"] = {"error": f"{type(exc).__name__}: {str(exc)[:200]}"}
    if world > 1 and not args.no_extras and C % world == 0 and wl["kind"] != "gmrf":
        # ---- strong scaling: the workload's chain count divided over the ranks (the weak line above grows it with N)
        Cs = C // world
        Ms, mss, _ = value_leg(ctx, wl, key, Cs, n, args.steps, args.warmup, thin, chain_offset=rank * Cs)
        extras["strong"] = {"value": Cs * world * args.steps / (mss * 1e-3), "unit": UNIT, "chains_total": Cs * world,
                            "chains_per_gpu": Cs, "ms_per_step": mss / args.steps, "scaling": "strong"}
        del Ms, _

    if rank == 0:
        roof = roofline_of(wl, C, n, p, op_ms, ms_max / args.steps, peaks, fp64_peak, syrk_ms, key=key)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": config_of(args, wl), "clocks": clk, "e2e": e2e,
            "gpu_launches": gpu_launches,
            "roofline": roof, "cpu_baseline": cpu_baseline, "ess": ess, "chains_failed": status_bad, "accept": accept,
        }
        line.update(extras)
        print(json.dumps(line), flush=True)
    if world > 1:
        ctx.dist.destroy_process_group()


def main():
    args = parse()
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, wl, args.workload)
    else:
        run_b200(args, wl, args.workload)


if __name__ == "__main__":
    main()
