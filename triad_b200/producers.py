"""Producers of the hot path's inputs (SURVEY.md §8 f3): the projection head shared by the reference's three
embedders and its patch dropout, each as one kernel.

``ProjectionHead``  src/model.py:32-34,68 (audio), :81-83,116 (text), :253-255,326 (visual):
    ``projection2(layer_norm(projection1(x)))``.  The module keeps the reference's attribute names and parameter
    shapes (``projection1`` / ``layer_norm`` / ``projection2``, so a checkpoint's ``state_dict`` loads unchanged);
    the forward is ONE launch of ``triad_project_tokens`` (tcgen05 GEMM -> LayerNorm epilogue -> tcgen05 GEMM ->
    bias / optional L2 normalisation), emitting the bf16 ``[B, N, D]`` K-major tensor the similarity kernel reads.
    The arithmetic follows the reference under autocast (bf16 GEMMs with fp32 accumulation, LayerNorm in fp32).
    Backward (training): ``triad_project_tokens_bwd``: one tcgen05 row pass recomputes the hidden activations
    from x (they are not stored) and writes the hidden gradient and the LayerNorm output, then the hand-written
    dense-gradient GEMMs form dx and the fp32 weight gradients; only the gradients autograd asks for are computed.

``patch_dropout``  src/model.py:268-308 without its per-image Python loop: the same ``torch.bernoulli`` call (same
    random stream, so the same output for the same seed), then ``triad_patch_compact`` moves the kept patches to
    the front of every image and zero-fills the rest.  The one host synchronisation left is the one that sizes the
    output (the batch's longest kept list), which the reference's ``max(...)`` needs too; the backward
    (``triad_patch_expand``) has none.

CUDA only, like the rest of the package: CPU tensors raise.
"""
from __future__ import annotations

import torch

from . import _lib, ops
from ._lib import check

HIDDEN = 512          # the reference hard-codes the head's hidden width (model.py:32, :81, :253)


def project_tokens(x: torch.Tensor, w1: torch.Tensor, b1: torch.Tensor, ln_g: torch.Tensor, ln_b: torch.Tensor, ln_eps: float,
                   w2: torch.Tensor, b2: torch.Tensor, normalize: bool = False) -> torch.Tensor:
    """Raw call: x (..., Din) bf16 -> (..., Dout) bf16."""
    lib = _lib.load()
    ops._require_cuda(x, w1, b1, ln_g, ln_b, w2, b2)
    if x.dtype != torch.bfloat16:
        raise TypeError("project_tokens computes in bf16 (the reference's autocast dtype); cast the encoder output first")
    Din = x.shape[-1]
    Dout = w2.shape[0]
    if w1.shape != (HIDDEN, Din) or w2.shape[1] != HIDDEN:
        raise ValueError(f"expected projection1 ({HIDDEN},{Din}) and projection2 (Dout,{HIDDEN}), got {tuple(w1.shape)} / {tuple(w2.shape)}")
    x2 = x.contiguous().view(-1, Din)
    M = x2.shape[0]
    w1b, w2b = w1.detach().to(torch.bfloat16).contiguous(), w2.detach().to(torch.bfloat16).contiguous()
    f32 = lambda t: t.detach().to(torch.float32).contiguous()                                         # noqa: E731
    b1f, gf, bf, b2f = f32(b1), f32(ln_g), f32(ln_b), f32(b2)
    out = torch.empty(M, Dout, dtype=torch.bfloat16, device=x.device)
    with ops._on(x):
        ws = ops._Workspace.get(lib.triad_project_workspace_bytes(), x.device, "project")
        check(lib.triad_project_tokens(x2.data_ptr(), w1b.data_ptr(), b1f.data_ptr(), gf.data_ptr(), bf.data_ptr(), float(ln_eps),
                                       w2b.data_ptr(), b2f.data_ptr(), M, Din, Dout, 1 if normalize else 0,
                                       out.data_ptr(), ws.data_ptr(), ws.numel(), ops._stream(x.device)), "triad_project_tokens")
    return out.view(*x.shape[:-1], Dout)


def project_tokens_bwd(x, w1, b1, ln_g, ln_b, ln_eps, w2, gy, need):
    """Raw call: gradients of ``project_tokens(..., normalize=False)`` for gy = dL/dout.  ``need`` is
    (x, w1, b1, ln_g, ln_b, w2, b2) booleans; returns the seven gradients (None where not needed): dx bf16 shaped
    like x, weight and bias gradients fp32."""
    lib = _lib.load()
    ops._require_cuda(x, w1, b1, ln_g, ln_b, w2, gy)
    Din, Dout = x.shape[-1], w2.shape[0]
    x2 = x.contiguous().view(-1, Din)
    M = x2.shape[0]
    gy2 = gy.to(torch.bfloat16).contiguous().view(M, Dout)
    w1b, w2b = w1.detach().to(torch.bfloat16).contiguous(), w2.detach().to(torch.bfloat16).contiguous()
    f32 = lambda t: t.detach().to(torch.float32).contiguous()                                         # noqa: E731
    b1f, gf, bf = f32(b1), f32(ln_g), f32(ln_b)
    dev = x.device
    out = lambda want, *shape, dtype=torch.float32: torch.empty(*shape, dtype=dtype, device=dev) if want else None  # noqa: E731
    dx = out(need[0], M, Din, dtype=torch.bfloat16)
    dw1, db1, dg, db = out(need[1], HIDDEN, Din), out(need[2], HIDDEN), out(need[3], HIDDEN), out(need[4], HIDDEN)
    dw2, db2 = out(need[5], Dout, HIDDEN), out(need[6], Dout)
    ptr = lambda t: t.data_ptr() if t is not None else None                                          # noqa: E731
    with ops._on(x):
        ws = ops._Workspace.get(lib.triad_project_tokens_bwd_workspace_bytes(M, Din, Dout), dev, "project_bwd")
        check(lib.triad_project_tokens_bwd(x2.data_ptr(), w1b.data_ptr(), b1f.data_ptr(), gf.data_ptr(), bf.data_ptr(),
                                           float(ln_eps), w2b.data_ptr(), gy2.data_ptr(), M, Din, Dout,
                                           ptr(dx), ptr(dw1), ptr(db1), ptr(dg), ptr(db), ptr(dw2), ptr(db2),
                                           ws.data_ptr(), ws.numel(), ops._stream(dev)), "triad_project_tokens_bwd")
    return (dx.view(x.shape) if dx is not None else None), dw1, db1, dg, db, dw2, db2


class _ProjectFn(torch.autograd.Function):
    """Forward: the fused kernel.  Backward: ``triad_project_tokens_bwd`` (the hidden activations are recomputed
    from x), computing only the gradients autograd asks for."""

    @staticmethod
    def forward(ctx, x, w1, b1, g, b, w2, b2, eps):
        ctx.save_for_backward(x, w1, b1, g, b, w2, b2)
        ctx.eps = eps
        return project_tokens(x, w1, b1, g, b, eps, w2, b2, normalize=False)

    @staticmethod
    def backward(ctx, gy):
        x, w1, b1, g, b, w2, b2 = ctx.saved_tensors
        need = ctx.needs_input_grad[:7]
        grads = project_tokens_bwd(x, w1, b1, g, b, ctx.eps, w2, gy, need)
        like = (x, w1, b1, g, b, w2, b2)
        return tuple(d.to(t.dtype) if d is not None else None for d, t in zip(grads, like)) + (None,)


class ProjectionHead(torch.nn.Module):
    """projection1 -> layer_norm -> projection2 of the reference's embedders, as one kernel.

    ``head(x)`` for x (B, N, Din) bf16 returns (B, N, embedding_dim) bf16; ``head.embed(x)`` additionally L2-normalises
    every token (retrieval.py:93-94)."""

    def __init__(self, in_features: int, embedding_dim: int = 512):
        super().__init__()
        self.projection1 = torch.nn.Linear(in_features, HIDDEN)
        self.layer_norm = torch.nn.LayerNorm(HIDDEN)
        self.projection2 = torch.nn.Linear(HIDDEN, embedding_dim)

    def _args(self):
        return (self.projection1.weight, self.projection1.bias, self.layer_norm.weight, self.layer_norm.bias,
                self.projection2.weight, self.projection2.bias)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        w1, b1, g, b, w2, b2 = self._args()
        if torch.is_grad_enabled() and (x.requires_grad or any(t.requires_grad for t in self._args())):
            return _ProjectFn.apply(x, w1, b1, g, b, w2, b2, self.layer_norm.eps)
        return project_tokens(x, w1, b1, g, b, self.layer_norm.eps, w2, b2, normalize=False)

    @torch.no_grad()
    def embed(self, x: torch.Tensor) -> torch.Tensor:
        w1, b1, g, b, w2, b2 = self._args()
        return project_tokens(x, w1, b1, g, b, self.layer_norm.eps, w2, b2, normalize=True)


class _PatchCompact(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, keep, max_len):
        lib = _lib.load()
        B, N, D = x.shape
        x = x.contiguous()
        keep8 = keep.to(torch.uint8).contiguous()
        out = torch.empty(B, max_len, D, dtype=x.dtype, device=x.device)
        with ops._on(x):
            check(lib.triad_patch_compact(x.data_ptr(), keep8.data_ptr(), B, N, D, x.element_size(), max_len, out.data_ptr(),
                                          ops._stream(x.device)), "triad_patch_compact")
        ctx.save_for_backward(keep8)
        ctx.n = N
        return out

    @staticmethod
    def backward(ctx, gy):
        (keep8,) = ctx.saved_tensors
        return patch_expand(gy, keep8, ctx.n), None, None


def patch_expand(gy: torch.Tensor, keep: torch.Tensor, n: int) -> torch.Tensor:
    """Backward of the compaction: (B, max_len, D) -> (B, n, D), row n of image b = gy[b, slot] where patch n is kept,
    zero elsewhere.  One launch, no host synchronisation."""
    lib = _lib.load()
    ops._require_cuda(gy, keep)
    B, L, D = gy.shape
    gy = gy.contiguous()
    keep8 = keep.to(torch.uint8).contiguous()
    gx = torch.empty(B, n, D, dtype=gy.dtype, device=gy.device)
    with ops._on(gy):
        check(lib.triad_patch_expand(gy.data_ptr(), keep8.data_ptr(), B, n, D, gy.element_size(), L, gx.data_ptr(),
                                     ops._stream(gy.device)), "triad_patch_expand")
    return gx


def patch_dropout(x: torch.Tensor, drop_rate: float, training: bool = True) -> torch.Tensor:
    """(B, N, D) -> (B, max_kept, D): kept patches compacted to the front of each image, zero rows behind.
    Differentiable w.r.t. ``x`` (gradients reach the kept patches only), like the reference's indexing."""
    if not training or drop_rate == 0:
        return x
    ops._require_cuda(x)
    B, N, D = x.shape
    keep = torch.bernoulli(torch.ones(B, N, device=x.device, dtype=x.dtype) * (1 - drop_rate)).bool()
    max_len = int(keep.sum(dim=1).max().item())                   # the one host synchronisation (output shape)
    return _PatchCompact.apply(x, keep, max_len)
