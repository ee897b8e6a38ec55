"""Time omc_nn_eigen_prep and omc_nn_eigen_draw at C2 size with CUDA events.

    python tools/perf_eigen_draw.py [C] [p]

Records from G = X'X / n + 0.1 I of random X (n = 4p).  The prep is timed once after one warm-up launch; the draw over
20 launches, each after a 256 MB write that flushes the L2, and once more with the records warm.  Bandwidth = the
bytes the draw must move (records read, beta and rss written) over its time.  One JSON line.
"""

import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from openmcmc_b200 import kernels as K  # noqa: E402


def main():
    C = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
    p = int(sys.argv[2]) if len(sys.argv) > 2 else 64
    K.init_device(0)
    dev, f64 = "cuda", torch.float64
    g = torch.Generator(device=dev).manual_seed(0)
    X = torch.randn(C, 4 * p, p, dtype=f64, device=dev, generator=g)
    G = X.transpose(1, 2) @ X / (4 * p) + 0.1 * torch.eye(p, dtype=f64, device=dev)
    stats = torch.cat([G.reshape(C, -1), torch.randn(C, p, dtype=f64, device=dev, generator=g),
                       torch.zeros(C, 2, dtype=f64, device=dev)], dim=1).contiguous()
    center = torch.cat([torch.randn(C, 2 * p, dtype=f64, device=dev, generator=g),
                        torch.ones(C, 2, dtype=f64, device=dev)], dim=1).contiguous()
    del X, G
    eig = torch.empty(C, K.eigen_record_len(p), dtype=f64, device=dev)
    mu0 = torch.zeros(p, dtype=f64, device=dev)

    def prep():
        K.nn_eigen_prep(C, p, stats, K.MAT_EYE, K.vec(None), K.vec(mu0), center, eig)

    prep()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    prep()
    e1.record()
    torch.cuda.synchronize()
    prep_ms = e0.elapsed_time(e1)

    tau = torch.full((C,), 1.0, dtype=f64, device=dev)
    lam = torch.full((C,), 0.01, dtype=f64, device=dev)
    beta = torch.empty(C, p, dtype=f64, device=dev)
    status = torch.zeros(C, dtype=torch.int32, device=dev)
    sweep = torch.zeros(1, dtype=torch.int64, device=dev)
    rng = K.rng(seed=1, sweep=sweep, site=1)

    def draw():
        K.nn_eigen_draw(C, p, eig, K.vec(tau, 1), K.vec(lam, 1), beta, rng, status=status, center=center,
                        rss_out=stats.data_ptr() + 8 * (p * p + p), rss_stride=p * p + p + 2)

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for _ in range(3):
        draw()
    flushed = []
    for k in range(20):
        flush.fill_(k & 255)
        e0.record()
        draw()
        e1.record()
        torch.cuda.synchronize()
        flushed.append(e0.elapsed_time(e1))
    e0.record()
    for _ in range(20):
        draw()
    e1.record()
    torch.cuda.synchronize()
    warm = e0.elapsed_time(e1) / 20
    ms = sorted(flushed)[len(flushed) // 2]
    nbytes = C * 8.0 * (K.eigen_record_len(p) + 1 + p + 1)
    print(json.dumps({"C": C, "p": p, "prep_ms": prep_ms, "draw_ms_flushed_median": ms, "draw_ms_flushed_min": min(flushed),
                      "draw_ms_warm": warm, "bytes": nbytes, "gbs_flushed": nbytes / (ms * 1e-3) / 1e9,
                      "status_bad": int(status.count_nonzero()), "finite": bool(torch.isfinite(beta).all())}))


if __name__ == "__main__":
    main()
