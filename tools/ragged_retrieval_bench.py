#!/usr/bin/env python
"""Top-k captions for one query image over a ragged caption gallery (RaggedGallery) against the same captions
zero-padded to [n, 77, D] and scored by the dense retrieve_topk.  The padded arm is a speed reference only: its
scores are wrong (padding joins the max in direction 0, direction 1 divides by 77).

Shape: 600 000 captions with cfg 3's lengths U[8, 77], D = 512, k = 10; query images of 256 and 1024 patches; both
directions.  The two arms are timed alternately in one process: device events around `iters` back-to-back calls,
the median of `reps` windows.  Reported per arm: ms per query (scores + top-k), the top-k alone, the bytes the
scorer reads (ragged: whole slots, gaps included; padded: 77 rows per caption) and the useful bytes (the captions'
own rows), GB/s over the bytes read, and TFLOP/s over the useful tokens (2 Nq D per token).  The card's name, power
limit and max SM clock are read in the same run.  Both galleries (26 GB and 47 GB) are far larger than L2.

With --fp8 the second arm is the same captions in an e4m3 RaggedGallery (one scale per slot row) instead of the
padded gallery; its bytes read are the slots' codes and scales, and the top-10 overlap is reported against the bf16
ragged arm.

    python tools/ragged_retrieval_bench.py [--captions 600000] [--iters 5] [--reps 5] [--fp8] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from triad_b200 import retrieval as R  # noqa: E402

D, K, T, LMAX = 512, 10, 0.07, 77


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


def build(n, dev, fp8, batch=50000):
    """(ragged gallery, second gallery, lengths) of the same random unit-norm captions, built batch by batch; the
    second gallery is the padded one [n, 77, D], or with fp8 an e4m3 RaggedGallery of the same bf16 rows."""
    lens = np.random.default_rng(3).integers(8, LMAX + 1, size=n)
    padded = None if fp8 else torch.zeros(n, LMAX, D, dtype=torch.bfloat16, device=dev)
    g = torch.Generator(device=dev).manual_seed(4)
    parts, parts8 = [], []
    for b0 in range(0, n, batch):
        lb = lens[b0:b0 + batch]
        flat = torch.nn.functional.normalize(torch.randn(int(lb.sum()), D, generator=g, device=dev), dim=1).bfloat16()
        mask = torch.arange(LMAX, device=dev)[None, :] < torch.from_numpy(lb).to(dev)[:, None]
        pb = torch.zeros(len(lb), LMAX, D, dtype=torch.bfloat16, device=dev) if fp8 else padded[b0:b0 + len(lb)]
        pb[mask] = flat
        parts.append(R.RaggedGallery.from_padded(pb, mask))
        if fp8:
            parts8.append(R.RaggedGallery.from_padded(pb, mask, fp8=True))
        del flat, pb
    return R.RaggedGallery.cat(parts), (R.RaggedGallery.cat(parts8) if fp8 else padded), lens


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--captions", type=int, default=600000)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--fp8", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ragged_retrieval_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    lines = []

    def emit(obj):
        print(json.dumps(obj), flush=True)
        lines.append(obj)

    emit({"card": card(), "torch": torch.__version__})
    ragged, other, lens = build(a.captions, dev, a.fp8)
    torch.cuda.synchronize()
    tokens = int(lens.sum())
    rows = ragged.n_slots * 256
    name2 = "ragged_fp8" if a.fp8 else "padded"
    emit({"captions": a.captions, "tokens": tokens, "mean_len": round(tokens / a.captions, 2), "slots": ragged.n_slots,
          "slot_rows_used": round(tokens / rows, 4), "ragged_GB": round(ragged.nbytes / 1e9, 2),
          name2 + "_GB": round((other.nbytes if a.fp8 else other.numel() * 2) / 1e9, 2)})
    read = {"ragged": rows * D * 2, name2: rows * (D + 4) if a.fp8 else a.captions * LMAX * D * 2}
    useful = {"ragged": tokens * D * 2, name2: tokens * (D + 4) if a.fp8 else tokens * D * 2}
    for Nq in (256, 1024):
        q = torch.nn.functional.normalize(torch.randn(Nq, D, device=dev), dim=1).bfloat16()
        Tt = torch.tensor(T, device=dev)
        for d in (0, 1):
            arms = {"ragged": ragged, name2: other}
            fns = {name: (lambda g=g: R.retrieve_topk(q, g, Tt, K, d)) for name, g in arms.items()}
            s_r = R._scores_ragged(q, ragged, Tt, d)
            topk_fn = lambda: R._topk(s_r, K)                              # noqa: E731
            for f in list(fns.values()) + [topk_fn]:
                f()
            torch.cuda.synchronize()
            times = {name: [] for name in fns}
            tk = []
            for _ in range(a.reps):
                for name, f in fns.items():                                # arms alternate within each repetition
                    times[name].append(window(f, a.iters))
                tk.append(window(topk_fn, a.iters))
            ids = {name: f()[1] for name, f in fns.items()}
            for name in fns:
                ms = statistics.median(times[name])
                emit({"arm": name, "Nq": Nq, "direction": d, "ms_per_query": round(ms, 3),
                      "ms_spread": [round(min(times[name]), 3), round(max(times[name]), 3)],
                      "bytes_read_GB": round(read[name] / 1e9, 2), "useful_GB": round(useful[name] / 1e9, 2),
                      "GB_per_s": round(read[name] / ms / 1e6, 1),
                      "useful_TFLOP_per_s": round(2.0 * Nq * tokens * D / ms / 1e9, 1)})
            emit({"topk_ms": round(statistics.median(tk), 3), "n": a.captions, "k": K, "Nq": Nq, "direction": d,
                  f"top10_overlap_with_{name2}": len(set(ids["ragged"].tolist()) & set(ids[name2].tolist()))})
            if a.fp8:
                ratio = statistics.median(times[name2]) / statistics.median(times["ragged"])
                emit({"Nq": Nq, "direction": d, "fp8_over_bf16_time": round(ratio, 3),
                      "fp8_over_bf16_bytes": round(read[name2] / read["ragged"], 3)})
            else:
                ratio = statistics.median(times["ragged"]) / statistics.median(times["padded"])
                emit({"Nq": Nq, "direction": d, "ragged_over_padded_time": round(ratio, 3),
                      "ragged_over_padded_bytes": round(read["ragged"] / read["padded"], 3)})
    emit({"card_after": card()})
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for obj in lines:
                f.write(json.dumps(obj) + "\n")


if __name__ == "__main__":
    main()
