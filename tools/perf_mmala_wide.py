"""Device time of one ManifoldMALA step above 64 parameters (mh.cu), with the n = 64 kernel beside it for reference.

    python tools/perf_mmala_wide.py [--reps 10] [--out FILE]

  - dense step (mmala_blocked_kernel) on 4096 chains at p = 96 / 128 / 136 / 137 / 256 / 512: a NORMAL_LINEAR term
    (regression record G | g | y'y | n, identity transform) plus a Normal prior with a dense precision; the record and
    the precision are shared by the chains (stride 0, L2-resident), the states are per chain;
  - element-wise step (mmala_diag_wide_kernel) on 8192 chains at n = 65 / 256 / 1024 / 4096: Poisson counts per chain
    with a Gamma(3, 1) prior;
  - p = n = 64 (mmala_kernel, the CTA-per-chain dense path) on the same two models.
Step size n^(-1/6).  Per shape: ms per step from CUDA events over `reps` launches after 2 warm-up launches.  Prints
the card's name, power limit and maximum SM clock first (same run).
"""
import argparse
import math
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from openmcmc_b200 import kernels as K  # noqa: E402


def timed(fn, reps):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def dense_problem(C, p, seed=1):
    g = torch.Generator(device="cuda").manual_seed(seed)
    f64, dev = torch.float64, "cuda"
    nd = 4 * p
    X = torch.randn(nd, p, dtype=f64, device=dev, generator=g) / math.sqrt(p)
    beta = 0.1 * torch.randn(p, dtype=f64, device=dev, generator=g)
    y = X @ beta + 0.2 * torch.randn(nd, dtype=f64, device=dev, generator=g)
    rec = torch.cat([(X.T @ X).reshape(-1), X.T @ y, (y @ y).reshape(1), torch.tensor([float(nd)], dtype=f64, device=dev)])
    B = torch.randn(p, p, dtype=f64, device=dev, generator=g)
    P = torch.eye(p, dtype=f64, device=dev) + B @ B.T / p
    tau, lam = torch.tensor([4.0], dtype=f64, device=dev), torch.tensor([1.0], dtype=f64, device=dev)
    logdet = torch.linalg.slogdet(P)[1].reshape(1)
    keep = [rec, P, tau, lam, logdet]
    terms = [K.term(K.TERM_NORMAL_LINEAR, stats=K.vec(rec), n_data=nd, scalar=K.vec(tau)),
             K.term(K.TERM_NORMAL_RESPONSE, mat_kind=K.MAT_DENSE, P=K.vec(P), scalar=K.vec(lam), logdet=K.vec(logdet))]
    theta = (beta + 0.05 * torch.randn(C, p, dtype=f64, device=dev, generator=g)).contiguous()
    return K.mh_model(C, p, terms), theta, keep


def elem_problem(C, n, seed=2):
    g = torch.Generator(device="cuda").manual_seed(seed)
    f64, dev = torch.float64, "cuda"
    k = torch.poisson(torch.full((C, n), 5.0, dtype=f64, device=dev), generator=g)
    a, b = torch.tensor([3.0], dtype=f64, device=dev), torch.tensor([1.0], dtype=f64, device=dev)
    keep = [k, a, b]
    terms = [K.term(K.TERM_POISSON_RATE, data=K.vec(k, n)), K.term(K.TERM_GAMMA_RESPONSE, p1=K.vec(a), p2=K.vec(b))]
    theta = ((k + 3.0) / 2.0).contiguous()
    return K.mh_model(C, n, terms), theta, keep


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    K.init_device()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    lines = [f"card: {gpu}  (name, power limit, max SM clock; read in this run)",
             f"torch {torch.__version__}, CUDA events over {args.reps} launches after 2 warm-up launches"]
    sweep = torch.zeros(1, dtype=torch.int64, device="cuda")

    def run(kind, C, n, step):
        model, theta, keep = (dense_problem if kind == "dense" else elem_problem)(C, n)
        ws_d = K.nn_dense_workspace(C, n) if kind == "dense" and n > 64 else 0
        ws = torch.empty(ws_d, dtype=torch.float64, device="cuda") if ws_d > 0 else None
        status = torch.zeros(C, dtype=torch.int32, device="cuda")
        counters = torch.zeros(C, 2, dtype=torch.int64, device="cuda")

        def fn():
            sweep.add_(1)
            K.mmala(model, theta, step, 0, K.rng(5, sweep=sweep), counters=counters, status=status, workspace=ws)

        ms = timed(fn, args.reps)
        c = counters.cpu()
        acc = float(c[:, 0].sum()) / max(1.0, float(c[:, 1].sum()))
        kern = ("mmala_kernel" if n <= 64 else
                "mmala_blocked_kernel<%s>" % ("global" if ws is not None else "shared") if kind == "dense"
                else "mmala_diag_wide_kernel")
        bad = int((status.cpu() & 3).ne(0).sum())
        lines.append(f"{kind:5s} C={C:5d} n={n:4d}  {kern:32s} {ms:9.3f} ms/step  {1e3 * ms / C:8.3f} us/chain-step  "
                     f"accept {acc:.2f}  chains flagged {bad}")
        print(lines[-1], flush=True)
        del keep

    # step n^(-1/6): a Langevin step that keeps part of the moves accepted as the dimension grows
    for p in (64, 96, 128, 136, 137, 256, 512):
        run("dense", 4096, p, p ** (-1.0 / 6.0))
    for n in (64, 65, 256, 1024, 4096):
        run("elem", 8192, n, n ** (-1.0 / 6.0))
    text = "\n".join(lines) + "\n"
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        open(args.out, "w").write(text)


if __name__ == "__main__":
    main()
