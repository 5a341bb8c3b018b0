"""Shared helpers for the parity tests (test infrastructure)."""
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

