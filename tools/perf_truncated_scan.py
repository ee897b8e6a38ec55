"""Device time of the truncated-prior NormalNormal scan for 64 < p <= 512 (trunc_scan.cu) at 4096 chains.

    python tools/perf_truncated_scan.py [--chains 4096] [--ps 65,128,256,512] [--reps 10]

Per shape: ms per scan (CUDA events over `reps` launches after 2 warm-up launches), record bytes / ms against the
7.7 TB/s HBM3e data-sheet figure, and the untruncated omc_nn_dense_draw (blocked Cholesky) on the same record for the
price of truncation.  Floors:
  - HBM: C (p^2 + p) 8 B / 7.7 TB/s (plus C p^2 8 B for a per-chain dense P0);
  - serial: the scan of ONE chain alone (one warp on an idle GPU) is p times the dependent latency of a coordinate
    (truncnorm + the x_i term); with W warps resident per SM the C chains run in ceil(C / (148 W)) rounds of that.
The records of 4096 chains are larger than the 126 MB L2 already at p = 65 (138 MB), so no flush is needed between
launches; the output says so.  Prints the card's name and power limit first.
"""
import argparse
import json
import math
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from openmcmc_b200 import kernels as K  # noqa: E402

HBM = 7.7e12
L2 = 126e6
WARPS_PER_SM = 12   # 4-warp CTAs, 134-168 registers per thread (profiles/r04_truncated_scan.txt, SASS summary)


def problem(C, p, dense, seed=1):
    g = torch.Generator(device="cuda").manual_seed(seed)
    dev, f64 = "cuda", torch.float64
    stats = torch.empty(C, p * p + p + 2, dtype=f64, device=dev)
    G = stats[:, : p * p].view(C, p, p)
    G.normal_(generator=g)
    G.add_(G.transpose(1, 2).clone()).mul_(0.05 / math.sqrt(p))
    G.diagonal(dim1=1, dim2=2).add_(2.0)
    stats[:, p * p:].normal_(generator=g)
    P0 = None
    if dense:
        P0 = torch.empty(C, p, p, dtype=f64, device=dev).normal_(generator=g)
        P0.add_(P0.transpose(1, 2).clone()).mul_(0.05 / math.sqrt(p))
        P0.diagonal(dim1=1, dim2=2).add_(1.0)
        P0 = P0.view(C, p * p)
    tau = torch.rand(C, dtype=f64, device=dev, generator=g) + 0.5
    lam = torch.rand(C, dtype=f64, device=dev, generator=g) + 0.1
    mu0 = torch.zeros(C, p, dtype=f64, device=dev)
    beta0 = 0.1 * torch.randn(C, p, dtype=f64, device=dev, generator=g)
    lo = torch.full((1,), -0.4, dtype=f64, device=dev)
    hi = torch.full((1,), 0.6, dtype=f64, device=dev)
    return dict(C=C, p=p, stats=stats, P0=P0, tau=tau, lam=lam, mu0=mu0, beta0=beta0, lo=lo, hi=hi)


def timed(fn, reps):
    fn()
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def run_shape(pr, reps, C=None, untruncated=True):
    C = pr["C"] if C is None else C
    p = pr["p"]
    kind = K.MAT_DENSE if pr["P0"] is not None else K.MAT_EYE
    pvec = K.vec(pr["P0"], p * p) if pr["P0"] is not None else K.vec(None)
    beta = pr["beta0"][:C].clone()
    status = torch.zeros(C, dtype=torch.int32, device="cuda")
    sweep = torch.zeros(1, dtype=torch.int64, device="cuda")
    args = (C, p, pr["stats"], K.vec(pr["tau"], 1), kind, pvec, K.vec(pr["lam"], 1), K.vec(pr["mu0"], p), beta,
            K.rng(seed=3, sweep=sweep, site=1))

    def scan():
        K.nn_dense_draw(*args, status=status, trunc=(K.vec(pr["lo"]), 1, K.vec(pr["hi"]), 1))

    out = {"ms": timed(scan, reps), "status_bad": int((status != 0).sum())}
    inside = bool(((beta >= -0.4) & (beta <= 0.6)).all())
    out["draws_inside_bounds"] = inside
    if untruncated:
        n = K.nn_dense_workspace(C, p)
        ws = torch.empty(n, dtype=torch.float64, device="cuda") if n else None

        def draw():
            K.nn_dense_draw(*args, status=status, workspace=ws)

        out["untruncated_ms"] = timed(draw, reps)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--chains", type=int, default=4096)
    ap.add_argument("--ps", default="65,128,256,512")
    ap.add_argument("--dense-p", type=int, default=256, help="p of the dense-prior case")
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print(f"# GPU: {gpu}")
    K.init_device(0)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    C = a.chains
    shapes = [(int(p), False) for p in a.ps.split(",")] + [(a.dense_p, True)]
    for p, dense in shapes:
        pr = problem(C, p, dense)
        rec_bytes = C * (p * p + p) * 8 + (C * p * p * 8 if dense else 0)
        r = run_shape(pr, a.reps)
        one = run_shape(pr, max(2, a.reps // 5), C=1, untruncated=False)
        wave = min(C, sms * WARPS_PER_SM)
        full = run_shape(pr, max(2, a.reps // 5), C=wave, untruncated=False)
        rounds = math.ceil(C / (sms * WARPS_PER_SM))
        hbm_floor = rec_bytes / HBM * 1e3
        serial_floor = rounds * one["ms"]
        print(json.dumps({
            "C": C, "p": p, "prior": "dense" if dense else "eye", "ms": round(r["ms"], 4),
            "record_MB": round(rec_bytes / 1e6, 1), "exceeds_L2": rec_bytes > L2,
            "GB_per_s": round(rec_bytes / r["ms"] / 1e6, 1), "frac_of_7.7TBps": round(hbm_floor / r["ms"], 4),
            "untruncated_draw_ms": round(r["untruncated_ms"], 4),
            "truncated_over_untruncated": round(r["ms"] / r["untruncated_ms"], 2),
            "one_chain_ms": round(one["ms"], 4), "us_per_coordinate_one_chain": round(one["ms"] / p * 1e3, 3),
            "one_wave_chains": wave, "one_wave_ms": round(full["ms"], 4), "rounds": rounds,
            "hbm_floor_ms": round(hbm_floor, 4), "serial_floor_ms": round(serial_floor, 4),
            "status_bad": r["status_bad"], "draws_inside_bounds": r["draws_inside_bounds"]}))
        del pr
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
