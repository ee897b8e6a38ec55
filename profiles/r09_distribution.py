"""Free-running C2 chains of two builds compared in distribution.

    python profiles/r09_distribution.py run TREE OUT.npz     # in the tree TREE (its bench.py and package)
    python profiles/r09_distribution.py compare A.npz B.npz

`run`: the C2 workload of bench.py (4096 chains, n = 10,000, p = 64, the same synthetic data), 200 burn-in sweeps and
1000 stored sweeps, then per chain and parameter element (beta, tau, lambda) the posterior mean, variance and ESS
(openmcmc_b200.diagnostics), the status bits and the sweep time.  `compare`: per chain and element the z-score of the
difference of the two posterior means over its Monte Carlo standard error sqrt(var_a / ess_a + var_b / ess_b); for two
samplers of the same posterior about 0.27 % of them lie beyond |z| > 3.
"""

import json
import os
import sys
import time

import numpy as np


def run(tree, out):
    sys.path.insert(0, tree)
    os.chdir(tree)
    import torch

    import bench
    from openmcmc_b200 import diagnostics as G
    from openmcmc_b200 import kernels as K
    from openmcmc_b200.mcmc import MCMC

    K.init_device(0)
    wl = bench.WORKLOADS["c2"]
    dev = torch.device("cuda", 0)
    mdl, samplers, state = bench.build_regression(wl["chains"], wl["n"], wl["p"], dev, 0, host=False)
    M = MCMC(state, samplers, model=mdl, n_burn=200, n_iter=1000, n_thin=1, n_chains=wl["chains"], seed=7,
             stream_store=False)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    M.run_mcmc()
    torch.cuda.synchronize()
    secs = time.perf_counter() - t0
    summ = G.summarize(M)
    res = {"status": M.status.cpu().numpy() if torch.is_tensor(M.status) else np.asarray(M.status), "seconds": secs}
    for name, v in summ.items():
        rec = v["records"].cpu().numpy()
        res[name + "_n"], res[name + "_mean"], res[name + "_var"], res[name + "_ess"] = (rec[:, :, 0], rec[:, :, 1],
                                                                                         rec[:, :, 2], rec[:, :, 3])
    np.savez(out, **res)
    print(json.dumps({"tree": tree, "seconds": secs, "status_nonzero": int(np.count_nonzero(res["status"]))}))


def compare(a_path, b_path):
    a, b = np.load(a_path), np.load(b_path)
    print(f"status bits set: A {int(np.count_nonzero(a['status']))} chains, B {int(np.count_nonzero(b['status']))} chains")
    allz = []
    for name in ("beta", "tau", "lambda"):
        ma, mb = a[name + "_mean"], b[name + "_mean"]
        va, vb = a[name + "_var"], b[name + "_var"]
        ea, eb = a[name + "_ess"], b[name + "_ess"]
        z = (ma - mb) / np.sqrt(va / ea + vb / eb)
        allz.append(z.ravel())
        n = a[name + "_n"][0, 0]
        print(f"{name:7s} elements {z.size:8d}  |z| > 3: {np.mean(np.abs(z) > 3) * 100:.3f} %  |z| > 4: "
              f"{np.mean(np.abs(z) > 4) * 100:.4f} %  mean z {np.mean(z):+.4f}  sd z {np.std(z):.4f}  "
              f"ESS per draw A {np.mean(ea) / n:.3f} B {np.mean(eb) / n:.3f}")
    z = np.concatenate(allz)
    print(f"all     elements {z.size:8d}  |z| > 3: {np.mean(np.abs(z) > 3) * 100:.3f} %  (normal: 0.270 %)")


if __name__ == "__main__":
    if sys.argv[1] == "run":
        run(os.path.abspath(sys.argv[2]), os.path.abspath(sys.argv[3]))
    else:
        compare(sys.argv[2], sys.argv[3])
