"""Shared helpers for the parity tests (test infrastructure)."""
import math
import os

import numpy as np
import torch

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    return dict(np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False))


def check_inputs_reproduce(gold, q, v):
    """The fixtures store checksums of the seeded inputs; a torch whose CPU generator differs
    would silently invalidate every comparison, so fail loudly instead."""
    assert abs(q.double().sum().item() - float(gold["in_q_sum"])) < 1e-9
    assert abs((q.double() ** 2).sum().item() - float(gold["in_q_sq"])) < 1e-9
    assert abs(v.double().sum().item() - float(gold["in_v_sum"])) < 1e-9
    assert abs((v.double() ** 2).sum().item() - float(gold["in_v_sq"])) < 1e-9


def _as64(x):
    if isinstance(x, torch.Tensor):
        return x.detach().to(device="cpu", dtype=torch.float64).reshape(-1)
    return torch.as_tensor(np.asarray(x), dtype=torch.float64).reshape(-1)


def rel_err(a, b):
    a, b = _as64(a), _as64(b)
    return ((a - b).norm() / b.norm().clamp(min=1e-30)).item()


def model_sims(raw, T, dtype):
    """The similarities S of the rounding model, from the exact dot products raw = <q, v> (fp64), returned in fp64.
    bf16 inputs: S = bf16(bf16(<q, v>) * T), as the reference computes them under autocast (the matmul rounds its fp32
    accumulator to bf16, the product with the fp32 temperature is rounded again; oracle.maxmean_forward).  fp32 inputs:
    S = T * <q, v>, unrounded."""
    if dtype == torch.bfloat16:
        T32 = torch.tensor(float(T), dtype=torch.float32, device=raw.device)
        return (raw.float().bfloat16().float() * T32).bfloat16().double()
    return raw * float(T)


def bf16_ulp(x):
    """One bf16 ulp of each element of x (fp64): 2^(floor(log2 |x|) - 7)."""
    return torch.exp2(torch.floor(torch.log2(x.abs().clamp(min=1e-30))) - 7)


def ambiguous_bf16_rounding(raw, sq, D, width=4.0):
    """True where an fp32 accumulator of the D-term dot product raw = <q, v> (fp64, exact) may round to bf16 either
    way: raw lies within `width` sigma of a bf16 rounding midpoint, sigma being the accumulator's random-walk rounding
    error 2^-24 * sqrt(D * <q^2, v^2>) (sq = <q^2, v^2>)."""
    acc_err = width * 2.0 ** -24 * math.sqrt(D) * sq.sqrt()
    a, r = raw.abs(), raw.float().bfloat16().double().abs()
    # the two midpoints around r; below a power of two the grid is twice as fine
    up, down = r + bf16_ulp(r) / 2, r - bf16_ulp(r * (1 - 2.0 ** -9)) / 2
    return torch.minimum((a - up).abs(), (a - down).abs()) < acc_err


def certify_near_ties(q, v, got, ref):
    """Argmax disagreements between two evaluations of the bf16 similarities, got and ref ((Bq, Bv, Nq) winner
    indices of q (Bq, Nq, D) against v (Bv, Nv, D)).  A disagreement is a genuine tie of the doubly rounded
    S = bf16(bf16(acc) * T) that the fp32 accumulation order can flip only when the two candidates' EXACT dot products
    (fp64) are less than 2 bf16 ulps of the accumulator apart.  (Two accumulators that round to the same or to ADJACENT
    bf16 values can land in the same output bin after the multiply by T moves them into the next binade, where the
    output grid is twice as coarse; anything further apart cannot tie.)  Returns (count, worst gap in ulps): the
    caller bounds both."""
    bad = (got != ref).nonzero()
    if bad.shape[0] == 0:
        return 0, 0.0
    i, j, a = bad.unbind(1)
    qa = q[i, a].double()
    x = (qa * v[j, got[i, j, a]].double()).sum(-1)
    y = (qa * v[j, ref[i, j, a]].double()).sum(-1)
    ulp = torch.exp2(torch.floor(torch.log2(torch.maximum(x.abs(), y.abs()).clamp(min=1e-300))) - 7)
    return int(bad.shape[0]), ((x - y).abs() / ulp).max().item()


def round_bf16_st(t):
    """t rounded to bf16 as a straight-through offset: the value is rounded, the gradient passes unchanged."""
    return t + (t.to(torch.bfloat16).double() - t).detach()


def head_fp64(x, w1, b1, g, b, w2, b2, eps, requires_grad=False):
    """fp64 evaluation of the projection head's autocast recipe: bf16 x / W1 / W2 / b1 / b2, h and ln rounded to bf16,
    fp32 LayerNorm parameters.  Returns the leaves (x, w1, b1, g, b, w2, b2 in fp64) and the intermediates: a = the
    first product plus bias before its rounding, h = bf16(a), y = the LayerNorm output before its rounding,
    ln = bf16(y) and out = ln . W2^T + bf16(b2) (not rounded)."""
    leaves = [x.double(), w1.bfloat16().double(), b1.double(), g.double(), b.double(), w2.bfloat16().double(), b2.double()]
    leaves = [t.detach().requires_grad_(requires_grad) for t in leaves]
    xx, ww1, bb1, gg, bb, ww2, bb2 = leaves
    a = xx.reshape(-1, xx.shape[-1]) @ ww1.t() + round_bf16_st(bb1)
    h = round_bf16_st(a)
    y = torch.nn.functional.layer_norm(h, (h.shape[-1],), gg, bb, eps)
    ln = round_bf16_st(y)
    out = ln @ ww2.t() + round_bf16_st(bb2)
    return leaves, {"a": a, "h": h, "y": y, "ln": ln, "out": out}


def head_fp64_grads(x, w1, b1, g, b, w2, b2, eps, gy):
    """Autograd in fp64 of head_fp64 for gy = dL/dout: the gradients of x, w1, b1, g, b, w2, b2."""
    leaves, t = head_fp64(x, w1, b1, g, b, w2, b2, eps, requires_grad=True)
    t["out"].backward(gy.reshape(t["out"].shape).double())
    return tuple(v.grad for v in leaves)

