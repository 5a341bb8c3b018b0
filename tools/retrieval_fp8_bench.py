#!/usr/bin/env python
"""BASELINE cfg 5 on an e4m3 gallery (Fp8Gallery) against the bf16 gallery: one query (text Nq = 77, audio Nq = 250)
against n_img images x 1024 patches x D = 512, max over patches, mean over tokens, top-10.

1. Both formats of the same random unit-norm gallery side by side (default 60 000 images: 63 GB bf16 + 31.6 GB fp8),
   timed alternately in the same process: ms/query, gallery GB/s (fp8: codes + scales), TFLOP/s, and the overlap of
   the two top-10s (synthetic data: not a recall figure).  Also the time of quantizing the gallery.
2. fp8 alone at 100 000 and 200 000 images (105 GB of codes at 200 000; the bf16 form, 210 GB, does not fit on one
   GPU).  These galleries repeat one 2 048-image random block (timing only: the data is far larger than L2).

The card's name and power limit are read in the same run.  Device events around `iters` back-to-back calls of
retrieve_topk, after a warm-up call per shape; the median of `reps` such windows is reported.

    python tools/retrieval_fp8_bench.py [--side 60000] [--big 100000,200000] [--iters 5] [--reps 5] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from triad_b200 import retrieval as R  # noqa: E402

NV, D, K, T = 1024, 512, 10, 1.5


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:                                   # noqa: BLE001
        out = f"nvidia-smi unavailable ({e})"
    return out


def window(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def random_fill(gal, g):
    step = max(1, (1 << 30) // (NV * D * 2))
    for i in range(0, gal.shape[0], step):
        blk = torch.randn(min(step, gal.shape[0] - i), NV, D, generator=g, device=gal.device)
        gal[i:i + blk.shape[0]] = torch.nn.functional.normalize(blk, dim=2).to(torch.bfloat16)


def row(fmt, n_img, Nq, ms, nbytes):
    flops = 2.0 * Nq * n_img * NV * D
    return {"format": fmt, "n_img": n_img, "Nq": Nq, "ms_per_query": round(ms, 3),
            "gallery_GB": round(nbytes / 1e9, 2), "gallery_GB_per_s": round(nbytes / ms / 1e6, 1),
            "TFLOP_per_s": round(flops / ms / 1e9, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--side", type=int, default=60000)
    ap.add_argument("--big", default="100000,200000")
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("retrieval_fp8_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    lines = []

    def emit(obj):
        s = json.dumps(obj)
        print(s, flush=True)
        lines.append(s)

    emit({"card": card(), "torch": torch.__version__, "Nv": NV, "D": D, "k": K, "iters": a.iters, "reps": a.reps})
    g = torch.Generator(device=dev).manual_seed(7)
    qs = {Nq: torch.nn.functional.normalize(torch.randn(Nq, D, generator=g, device=dev), dim=1).to(torch.bfloat16)
          for Nq in (77, 250)}

    # ---- 1. bf16 and fp8 side by side ----
    if a.side > 0:
        n = a.side
        t0 = time.time()
        bf = torch.empty(n, NV, D, dtype=torch.bfloat16, device=dev)
        random_fill(bf, g)
        torch.cuda.synchronize()
        fill_s = time.time() - t0
        f8 = R.Fp8Gallery.empty(n, NV, D, device=dev)
        f8.put(0, bf[:1])                                     # warm-up of the quantizer
        torch.cuda.synchronize()
        qms = window(lambda: f8.put(0, bf), 1)
        emit({"side_by_side_gallery": n, "bf16_GB": round(bf.numel() * 2 / 1e9, 2), "fp8_GB": round(f8.nbytes / 1e9, 2),
              "fill_s": round(fill_s, 1), "quantize_ms": round(qms, 2),
              "quantize_GB_per_s": round((bf.numel() * 2 + f8.nbytes) / qms / 1e6, 1)})
        for Nq, q in qs.items():
            R.retrieve_topk(q, bf, T, K)
            R.retrieve_topk(q, f8, T, K)
            torch.cuda.synchronize()
            tb, tf = [], []
            for _ in range(a.reps):
                tb.append(window(lambda: R.retrieve_topk(q, bf, T, K), a.iters))
                tf.append(window(lambda: R.retrieve_topk(q, f8, T, K), a.iters))
            sb, ib = R.retrieve_topk(q, bf, T, K)
            sf, i8 = R.retrieve_topk(q, f8, T, K)
            mb, mf = statistics.median(tb), statistics.median(tf)
            rb, rf = row("bf16", n, Nq, mb, bf.numel() * 2), row("fp8", n, Nq, mf, f8.nbytes)
            rb["spread_ms"] = [round(min(tb), 3), round(max(tb), 3)]
            rf["spread_ms"] = [round(min(tf), 3), round(max(tf), 3)]
            emit(rb)
            emit(rf)
            emit({"Nq": Nq, "n_img": n, "fp8_speedup": round(mb / mf, 3),
                  "top10_overlap": len(set(ib.tolist()) & set(i8.tolist())),
                  "top1_bf16": [int(ib[0]), round(float(sb[0]), 5)], "top1_fp8": [int(i8[0]), round(float(sf[0]), 5)]})
        del bf, f8
        torch.cuda.empty_cache()

    # ---- 2. fp8 alone on large galleries ----
    for n in [int(x) for x in a.big.split(",") if x]:
        free, total = torch.cuda.mem_get_info(dev)
        f8 = R.Fp8Gallery.empty(n, NV, D, device=dev)
        blk = 2048
        src = torch.empty(blk, NV, D, dtype=torch.bfloat16, device=dev)
        random_fill(src, g)
        f8.put(0, src)
        del src
        for i in range(blk, n, blk):
            b = min(blk, n - i)
            f8.codes[i:i + b].view(torch.uint8).copy_(f8.codes[:b].view(torch.uint8))
            f8.scales[i:i + b].copy_(f8.scales[:b])
        torch.cuda.synchronize()
        emit({"fp8_alone_gallery": n, "fp8_GB": round(f8.nbytes / 1e9, 2), "bf16_would_be_GB": round(n * NV * D * 2 / 1e9, 2),
              "device_free_GB_before": round(free / 1e9, 1), "device_total_GB": round(total / 1e9, 1)})
        for Nq, q in qs.items():
            R.retrieve_topk(q, f8, T, K)
            torch.cuda.synchronize()
            tf = [window(lambda: R.retrieve_topk(q, f8, T, K), a.iters) for _ in range(a.reps)]
            r = row("fp8", n, Nq, statistics.median(tf), f8.nbytes)
            r["spread_ms"] = [round(min(tf), 3), round(max(tf), 3)]
            emit(r)
        del f8
        torch.cuda.empty_cache()

    emit({"card_after": card()})
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
