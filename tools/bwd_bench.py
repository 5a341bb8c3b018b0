#!/usr/bin/env python
"""Times the pieces of one step at a BASELINE shape and cross-checks the backward variants.

    python tools/bwd_bench.py [cfg2|cfg3|...] [iters] [Bq] [Bv] [Nv]

Bq defaults to the config's batch, Bv to Bq, and Nv (patches per image) to the config's.

Prints CUDA-event times of: forward, InfoNCE, dq (tiled / generic), dv (default / generic), and
the max relative difference between the variants' outputs (they must agree to bf16 rounding).
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402
from triad_b200 import _lib, ops  # noqa: E402


def timeit(fn, iters):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def rel(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return ((a - b).norm() / b.norm().clamp(min=1e-30)).item()


def main():
    cfg = dict(bench.CONFIGS[sys.argv[1] if len(sys.argv) > 1 else "cfg2"])
    iters = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    Bq = int(sys.argv[3]) if len(sys.argv) > 3 else cfg["B"]       # local query rows (a rank's shard)
    Bv = int(sys.argv[4]) if len(sys.argv) > 4 else Bq             # images (the all-gathered batch)
    if len(sys.argv) > 5:
        cfg["Nv"] = int(sys.argv[5])
    dev = torch.device("cuda", 0)
    (q, _, mask), = bench.make_device_inputs(cfg, Bq, 1234, dev, 1)
    (_, v, _), = bench.make_device_inputs(cfg, Bv, 4321, dev, 1)
    _, Nq, D = q.shape
    Nv = v.shape[1]
    B = Bv
    scale = ops.row_scale(mask, Bq, Nq, dev)
    T = torch.tensor(1.5, device=dev)
    clip, idx = ops.maxmean_fwd(q, v, scale, T)
    row_lse, col_part = ops.infonce_partial(clip, B, 0)
    g, sums = ops.infonce_finish(clip, B, 0, row_lse, col_part.reshape(1, 2, B))
    print(f"shape Bq={Bq} Bv={Bv} Nq={Nq} Nv={Nv} D={D} masked={mask is not None}  block loss sum={sums[0].item() / (2 * B):.6f}")

    pack_f = _lib.FWD_PACK_ROWS if mask is not None else 0        # what the drop-in does for masked bf16 queries
    pack_b = _lib.BWD_PACK_ROWS if mask is not None else 0
    if mask is not None:
        t_unp = timeit(lambda: ops.maxmean_fwd(q, v, scale, T), iters)
        print(f"fwd without row packing {t_unp:.3f} ms")
        clip_p, idx_p = ops.maxmean_fwd(q, v, scale, T, flags=pack_f)
        print("packed vs unpacked clip exact:", torch.equal(clip_p, clip))
    t_fwd = timeit(lambda: ops.maxmean_fwd(q, v, scale, T, flags=pack_f), iters)
    t_nce = timeit(lambda: ops.infonce_finish(clip, B, 0, *ops.infonce_partial(clip, B, 0)[:1],
                                               col_part.reshape(1, 2, B)), iters)
    tf = 2.0 * Bv * (mask.sum().item() if mask is not None else Bq * Nq) * Nv * D / 1e12
    print(f"fwd {t_fwd:.3f} ms ({tf / t_fwd * 1e3:.0f} TFLOP/s)   infonce {t_nce:.3f} ms")

    def bwd(dq, dv, flags):
        return ops.maxmean_bwd(q, v, idx, g, clip, scale, T, need_dq=dq, need_dv=dv, need_dT=False, flags=flags)

    outs = {}
    for name, dq_, dv_, fl in (("dq tiled", True, False, pack_b), ("dq unpacked", True, False, 0),
                               ("dq generic", True, False, _lib.BWD_GENERIC_DQ),
                               ("dv default", False, True, 0), ("dv generic", False, True, _lib.BWD_GENERIC_DV)):
        t = timeit(lambda: bwd(dq_, dv_, fl), iters)
        o = bwd(dq_, dv_, fl)
        outs[name] = o[0] if dq_ else o[1]
        print(f"{name:12s} {t:.3f} ms")
    torch.cuda.synchronize()
    print("dq tiled vs generic  rel diff", rel(outs["dq tiled"], outs["dq generic"]),
          " exact:", torch.equal(outs["dq tiled"], outs["dq generic"]))
    print("dv default vs generic rel diff", rel(outs["dv default"], outs["dv generic"]),
          " exact:", torch.equal(outs["dv default"], outs["dv generic"]))
    t_all = timeit(lambda: ops.maxmean_bwd(q, v, idx, g, clip, scale, T, flags=pack_b), iters)
    tot = t_fwd + t_nce + t_all
    print(f"bwd (dq+dv+dT) {t_all:.3f} ms    fwd+nce+bwd {tot:.3f} ms  = {Bq * Bv / tot / 1e3:.2f} M pairs/s per GPU")


if __name__ == "__main__":
    main()
