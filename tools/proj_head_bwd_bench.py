"""Forward + backward of ProjectionHead at the reference's three producer shapes, three arms:

  kernels      ProjectionHead: triad_project_tokens forward, triad_project_tokens_bwd backward
  closed_form  the same forward with the torch closed-form backward the kernels replaced (bf16 library GEMMs and
               ~25 elementwise ATen kernels over fp32 [M, 512] temporaries; kept here as the comparison arm)
  torch_nn     projection2(layer_norm(projection1(x))) from torch.nn modules under bf16 autocast

CUDA events around every iteration; every shape and arm is warmed up first, and the arms alternate inside the timed
loop (each round runs every arm once, in a rotating order).  At each shape the arms' gradients are compared before
timing.  The working set of one iteration (x, gy, the gradients, the temporaries) exceeds the 126 MB L2 at the audio
and visual shapes; nothing is flushed between iterations.

    python tools/proj_head_bwd_bench.py [--iters 30] [--warmup 5] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from triad_b200.producers import ProjectionHead, project_tokens  # noqa: E402

SHAPES = {"audio_cfg2": (256, 250, 768, 512), "visual": (256, 256, 768, 512), "text": (512, 77, 768, 512)}


class _ClosedFormFn(torch.autograd.Function):
    """The kernel forward with the retired closed-form backward."""

    @staticmethod
    def forward(ctx, x, w1, b1, g, b, w2, b2, eps):
        ctx.save_for_backward(x, w1, b1, g, b, w2)
        ctx.eps = eps
        return project_tokens(x, w1, b1, g, b, eps, w2, b2, normalize=False)

    @staticmethod
    def backward(ctx, gy):
        x, w1, b1, g, b, w2 = ctx.saved_tensors
        Din = x.shape[-1]
        x2 = x.reshape(-1, Din)
        gy2 = gy.reshape(-1, gy.shape[-1]).to(torch.bfloat16)
        w1b, w2b = w1.to(torch.bfloat16), w2.to(torch.bfloat16)
        h = (x2 @ w1b.t() + b1.to(torch.bfloat16)).float()
        mu = h.mean(dim=1, keepdim=True)
        rstd = torch.rsqrt(h.var(dim=1, unbiased=False, keepdim=True) + ctx.eps)
        xh = (h - mu) * rstd
        ln = (xh * g.float() + b.float()).to(torch.bfloat16)
        gw2 = gy2.t() @ ln
        gb2 = gy2.float().sum(dim=0)
        gln = (gy2 @ w2b).float()
        gg = (gln * xh).sum(dim=0)
        gb = gln.sum(dim=0)
        gxh = gln * g.float()
        gh = (gxh - gxh.mean(dim=1, keepdim=True) - xh * (gxh * xh).mean(dim=1, keepdim=True)) * rstd
        ghb = gh.to(torch.bfloat16)
        gw1 = ghb.t() @ x2
        gb1 = gh.sum(dim=0)
        gx = (ghb @ w1b).view_as(x)
        return gx, gw1.to(w1.dtype), gb1.to(b1.dtype), gg.to(g.dtype), gb.to(b.dtype), gw2.to(w2.dtype), gb2.to(b1.dtype), None


def _args(h):
    return (h.projection1.weight, h.projection1.bias, h.layer_norm.weight, h.layer_norm.bias,
            h.projection2.weight, h.projection2.bias)


def _run(arm, head, x):
    if arm == "kernels":
        return head(x)
    if arm == "closed_form":
        return _ClosedFormFn.apply(x, *_args(head), head.layer_norm.eps)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        return head.projection2(head.layer_norm(head.projection1(x)))


def _grads(arm, head, x, gy):
    head.zero_grad(set_to_none=True)
    x.grad = None
    _run(arm, head, x).backward(gy)
    return [x.grad] + [p.grad for p in _args(head)]


def _rel(a, b):
    a, b = a.double(), b.double()
    return ((a - b).norm() / b.norm().clamp(min=1e-30)).item()


def card():
    name = torch.cuda.get_device_name()
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                             str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (no CPU timing)")
    name, pl = card()
    lines = [f"device: {name}; power.limit, clocks.max.sm: {pl}",
             f"ProjectionHead forward + backward, CUDA events, {a.iters} alternating rounds after {a.warmup} warm-up rounds; ms per call"]
    arms = ("kernels", "closed_form", "torch_nn")
    results = {}
    for sname, (B, N, Din, Dout) in SHAPES.items():
        torch.manual_seed(0)
        head = ProjectionHead(Din, Dout).cuda()
        with torch.no_grad():
            head.layer_norm.weight.uniform_(0.5, 1.5)
            head.layer_norm.bias.uniform_(-0.3, 0.3)
        x = torch.randn(B, N, Din, device="cuda").bfloat16().requires_grad_()
        gy = (torch.randn(B, N, Dout, device="cuda") * 0.05).bfloat16()
        # gradients agree at the timed size
        g = {arm: _grads(arm, head, x, gy) for arm in arms}
        agree = {f"{arm}_vs_closed_form": max(_rel(u, v) for u, v in zip(g[arm], g["closed_form"])) for arm in ("kernels", "torch_nn")}
        del g
        for _ in range(a.warmup):
            for arm in arms:
                _grads(arm, head, x, gy)
        torch.cuda.synchronize()
        fwd = {arm: 0.0 for arm in arms}
        tot = {arm: 0.0 for arm in arms}
        for it in range(a.iters):
            order = arms[it % 3:] + arms[:it % 3]
            for arm in order:
                head.zero_grad(set_to_none=True)
                x.grad = None
                e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                e0.record()
                y = _run(arm, head, x)
                e1.record()
                y.backward(gy)
                e2.record()
                e2.synchronize()
                fwd[arm] += e0.elapsed_time(e1)
                tot[arm] += e0.elapsed_time(e2)
        res = {arm: {"fwd_bwd_ms": tot[arm] / a.iters, "bwd_ms": (tot[arm] - fwd[arm]) / a.iters} for arm in arms}
        results[sname] = {"shape": [B, N, Din, Dout], "arms": res, "max_rel_grad_diff": agree}
        lines.append(f"{sname} B={B} N={N} Din={Din} Dout={Dout} (M={B * N}):")
        for arm in arms:
            lines.append(f"  {arm:12s} fwd+bwd {res[arm]['fwd_bwd_ms']:8.3f}   bwd {res[arm]['bwd_ms']:8.3f}")
        lines.append("  max relative gradient difference vs closed_form: " + ", ".join(f"{k} {v:.2e}" for k, v in agree.items()))
        del head, x, gy
        torch.cuda.empty_cache()
    text = "\n".join(lines)
    print(text)
    print(json.dumps({"device": name, "power_limit": pl, "results": results}))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n" + json.dumps({"device": name, "power_limit": pl, "results": results}) + "\n")


if __name__ == "__main__":
    main()
