#!/usr/bin/env python
"""Where the dense-regulariser forward's time goes at cfg 2: plain forward, regulariser-only pass with / without the
N stores, the merged pass, and the raw write bandwidth of the same 8.4 GB (memset / fill)."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import bench  # noqa: E402
from triad_b200 import ops  # noqa: E402
from triad_b200 import regularizers as R  # noqa: E402


def timed(fn, n=5):
    fn(); torch.cuda.synchronize()
    ts = []
    for _ in range(n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return min(ts), sum(ts) / len(ts)


def main():
    cfg = bench.CONFIGS[sys.argv[1] if len(sys.argv) > 1 else "cfg2"]
    dev = torch.device("cuda", 0)
    (q, v, _), = bench.make_device_inputs(cfg, cfg["B"], 1234, dev, 1)
    B, Nq, Nv = cfg["B"], cfg["Nq"], cfg["Nv"]
    T = torch.tensor(1.5, device=dev)
    scale = ops.row_scale(None, B, Nq, dev)
    coef = 2.0 / (float(B * Nq) * B * Nv)
    sums = torch.zeros(2, dtype=torch.float64, device=dev)
    N = torch.empty(B * Nq, B * Nv, dtype=torch.bfloat16, device=dev)
    print("plain forward          ", timed(lambda: ops.maxmean_fwd(q, v, scale, T)))
    print("regulariser, no stores ", timed(lambda: R.nonneg_fused_chunk(q, v, T, -60.0, coef, False, sums)))
    print("regulariser, stores    ", timed(lambda: R.nonneg_fused_chunk(q, v, T, -60.0, coef, True, sums)))
    print("merged                 ", timed(lambda: ops.maxmean_fwd_nonneg(q, v, scale, T, -60.0, coef)))
    print("zero_ of N (%.1f GB)    " % (N.numel() * 2 / 1e9), timed(lambda: N.zero_()))
    print("fill_ of N             ", timed(lambda: N.fill_(1.0)))
    M = torch.empty_like(N)
    print("copy_ N -> M           ", timed(lambda: M.copy_(N)))


if __name__ == "__main__" and not (len(sys.argv) > 1 and sys.argv[1] == "gemms"):
    main()


def gemms():
    """The two backward GEMMs at cfg 2: hand-written (triad_dense_grad_gemm) vs the library."""
    dev = torch.device("cuda", 0)
    cfg = bench.CONFIGS[sys.argv[2] if len(sys.argv) > 2 else "cfg2"]
    (q, v, _), = bench.make_device_inputs(cfg, cfg["B"], 1234, dev, 1)
    B, Nq, Nv, D = cfg["B"], cfg["Nq"], cfg["Nv"], cfg["D"]
    N = (torch.randn(B * Nq, B * Nv, device=dev, dtype=torch.bfloat16) * 0.01)
    q2, v2 = q.view(-1, D), v.view(-1, D)
    print("dQ = N V     own  ", timed(lambda: ops.dense_grad_gemm(N, v2, 0)))
    print("dQ = N V     torch", timed(lambda: torch.mm(N, v2)))
    print("dV = N^T Q   own  ", timed(lambda: ops.dense_grad_gemm(N, q2, 1)))
    print("dV = N^T Q   torch", timed(lambda: torch.mm(N.t(), q2)))
    a, b = ops.dense_grad_gemm(N, v2, 0), torch.mm(N, v2)
    print("rel diff dQ", ((a.float() - b.float()).norm() / b.float().norm()).item())
    a, b = ops.dense_grad_gemm(N, q2, 1), torch.mm(N.t(), q2)
    print("rel diff dV", ((a.float() - b.float()).norm() / b.float().norm()).item())


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "gemms":
    gemms()
