"""Quick device-time probe of omc_nn_dense_draw at the C2 shape (4096 chains, p = 64), with a torch fp64 check of the
posterior mean (not the bench; used while tuning)."""
import json
import sys

import torch

sys.path.insert(0, ".")
from openmcmc_b200 import kernels as K

K.init_device(0)
C = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
p = int(sys.argv[2]) if len(sys.argv) > 2 else 64
g = torch.Generator(device="cuda").manual_seed(1)
A = torch.randn(C, 4 * p, p, dtype=torch.float64, device="cuda", generator=g)
G = A.transpose(1, 2) @ A
gv = torch.randn(C, p, dtype=torch.float64, device="cuda", generator=g)
stats = torch.cat([G.reshape(C, -1), gv, torch.zeros(C, 2, dtype=torch.float64, device="cuda")], dim=1).contiguous()
tau = torch.rand(C, dtype=torch.float64, device="cuda", generator=g) + 0.5
lam = torch.rand(C, dtype=torch.float64, device="cuda", generator=g) + 0.1
mu0 = torch.zeros(p, dtype=torch.float64, device="cuda")
beta = torch.empty(C, p, dtype=torch.float64, device="cuda")
pmu = torch.empty(C, p, dtype=torch.float64, device="cuda")
sweep = torch.zeros(1, dtype=torch.int64, device="cuda")
status = torch.zeros(C, dtype=torch.int32, device="cuda")
_ws = K.nn_dense_workspace(C, p)
ws = torch.empty(_ws, dtype=torch.float64, device="cuda") if _ws else None


def call(probe=None):
    K.nn_dense_draw(C, p, stats, K.vec(tau, 1), K.MAT_EYE, K.vec(None), K.vec(lam, 1), K.vec(mu0, 0), beta,
                    K.rng(seed=1, sweep=sweep, site=3), probe_mu=probe, status=status, workspace=ws)


call(pmu)
torch.cuda.synchronize()
Q = lam.view(C, 1, 1) * torch.eye(p, dtype=torch.float64, device="cuda") + tau.view(C, 1, 1) * G
ref = torch.linalg.solve(Q, (tau.view(C, 1) * gv).unsqueeze(-1)).squeeze(-1)
err = float(((pmu - ref).abs().amax(dim=1) / ref.abs().amax(dim=1)).max())
for _ in range(3):
    call()
torch.cuda.synchronize()
reps = 20
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(reps):
    call()
e1.record()
torch.cuda.synchronize()
print(json.dumps({"C": C, "p": p, "ms": e0.elapsed_time(e1) / reps, "mean_rel_err_vs_torch": err,
                  "status_bad": int((status != 0).sum())}))
