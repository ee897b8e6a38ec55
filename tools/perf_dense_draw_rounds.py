"""Device time of omc_nn_dense_draw (left-looking warp kernel, 40 < p <= 64) by chain count, one JSON line per (p, C):

    python tools/perf_dense_draw_rounds.py [P ...]          (default: 48 56 63 64)

Chain counts: 4096 (C2), C = 148 w for w = 1, 2, 4, 7, 14 (one round of the persistent warps: the launch packs them
into ceil(C / 14) CTAs of up to 14 warps, one per SM), and C = w (a single CTA of w warps on one SM: the time of one
chain with w - 1 others sharing the SM's schedulers).  Whether that time grows with w says whether one chain is
limited by its dependent latency (flat) or by the issue slots it shares (growing).  Records are warm in L2; the same
inputs as tools/perf_dense_draw.py.  OMC_LIB selects the library, as for the other tools.
"""
import json
import sys

import torch

sys.path.insert(0, ".")
from openmcmc_b200 import kernels as K  # noqa: E402

K.init_device(0)
PS = [int(a) for a in sys.argv[1:]] or [48, 56, 63, 64]
WS = [1, 2, 4, 7, 14]
CS = [4096] + [148 * w for w in WS] + WS


def setup(C, p):
    g = torch.Generator(device="cuda").manual_seed(1)
    A = torch.randn(C, 4 * p, p, dtype=torch.float64, device="cuda", generator=g)
    G = A.transpose(1, 2) @ A
    gv = torch.randn(C, p, dtype=torch.float64, device="cuda", generator=g)
    stats = torch.cat([G.reshape(C, -1), gv, torch.zeros(C, 2, dtype=torch.float64, device="cuda")], dim=1).contiguous()
    tau = torch.rand(C, dtype=torch.float64, device="cuda", generator=g) + 0.5
    lam = torch.rand(C, dtype=torch.float64, device="cuda", generator=g) + 0.1
    mu0 = torch.zeros(p, dtype=torch.float64, device="cuda")
    beta = torch.empty(C, p, dtype=torch.float64, device="cuda")
    sweep = torch.zeros(1, dtype=torch.int64, device="cuda")
    status = torch.zeros(C, dtype=torch.int32, device="cuda")

    def call():
        K.nn_dense_draw(C, p, stats, K.vec(tau, 1), K.MAT_EYE, K.vec(None), K.vec(lam, 1), K.vec(mu0, 0), beta,
                        K.rng(seed=1, sweep=sweep, site=3), status=status)
    return call, status


for p in PS:
    for C in CS:
        call, status = setup(C, p)
        for _ in range(5):
            call()
        torch.cuda.synchronize()
        reps = 200
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            call()
        e1.record()
        torch.cuda.synchronize()
        print(json.dumps({"p": p, "C": C, "ms": round(e0.elapsed_time(e1) / reps, 5), "status_bad": int((status != 0).sum())}),
              flush=True)
