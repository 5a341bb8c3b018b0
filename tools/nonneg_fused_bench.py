#!/usr/bin/env python
"""Times the dense-regulariser mode of the tcgen05 forward (triad_nonneg_fused_chunk) in 64-image launches, with and
without the N stores, next to the normal forward split into the same launches.

    python tools/nonneg_fused_bench.py [cfg2|cfg3|...]
"""
import sys, torch
import os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
from triad_b200 import regularizers as R, ops
cfg = bench.CONFIGS[sys.argv[1] if len(sys.argv) > 1 else "cfg2"]
B, Nq = cfg["B"], cfg["Nq"]
dev = torch.device("cuda", 0)
(q, v, _), = bench.make_device_inputs(cfg, B, 1, dev, 1)
T = torch.tensor(1.5, device=dev)
sums = torch.zeros(2, dtype=torch.float64, device=dev)
def run(write):
    for j0 in range(0, B, 64):
        R.nonneg_fused_chunk(q, v[j0:j0+64], T, -60.0, 1e-9, write, sums)
for write in (False, True):
    run(write); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10): run(write)
    e1.record(); torch.cuda.synchronize()
    print("write_n", write, e0.elapsed_time(e1) / 10, "ms per full pass")
scale = ops.row_scale(None, B, Nq, dev)
def fwd_chunks():
    for j0 in range(0, B, 64):
        ops.maxmean_fwd(q, v[j0:j0+64], scale, T)
fwd_chunks(); torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(10): fwd_chunks()
e1.record(); torch.cuda.synchronize()
print(f"normal forward as {(B + 63) // 64} launches of 64 images:", e0.elapsed_time(e1) / 10, "ms")
