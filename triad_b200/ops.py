"""torch-facing wrappers of the C ABI: raw calls, a grow-only workspace cache and the two
autograd Functions (max-mean similarity, symmetric InfoNCE) the drop-in methods are built from.

PyTorch is plumbing here (device memory, streams, autograd bookkeeping); every arithmetic
step of the path runs in libtriad_b200.so.
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import torch

from . import _lib
from ._lib import check

_DT = {torch.float32: _lib.DTYPE_F32, torch.bfloat16: _lib.DTYPE_BF16}


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _stream(device=None) -> int:
    """Raw handle of torch's current stream ON `device` (the tensors' device, not the process-wide current one)."""
    return torch.cuda.current_stream(device).cuda_stream


def _on(t: torch.Tensor):
    """Device guard for one library call: the kernels are launched on the device that owns `t`, whatever the
    process-wide current device is (several GPUs in one process, autograd's backward threads)."""
    return torch.cuda.device(t.device)


def _require_cuda(*ts: torch.Tensor) -> None:
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("triad_b200 runs on CUDA tensors only (there is no CPU fallback)")


class _Workspace:
    """One grow-only byte buffer per (device, stream, tag)."""
    _bufs: Dict[Tuple, torch.Tensor] = {}

    @classmethod
    def get(cls, nbytes: int, device: torch.device, tag: str) -> torch.Tensor:
        key = (device.index, _stream(device), tag)
        buf = cls._bufs.get(key)
        if buf is None or buf.numel() < nbytes:
            buf = torch.empty(max(nbytes, 1024), dtype=torch.uint8, device=device)
            cls._bufs[key] = buf
        return buf


def _dtype_code(t: torch.Tensor) -> int:
    try:
        return _DT[t.dtype]
    except KeyError:
        raise TypeError(f"triad_b200 supports float32 and bfloat16 embeddings, got {t.dtype}") from None


def temperature_tensor(temperature, device) -> torch.Tensor:
    """The kernels read the temperature from device memory (no host sync on the nn.Parameter)."""
    if isinstance(temperature, torch.Tensor):
        t = temperature.detach() if temperature.requires_grad else temperature
        if t.dtype != torch.float32 or t.device != device or t.numel() != 1:
            t = t.to(device=device, dtype=torch.float32).reshape(())
        return t
    return torch.tensor(float(temperature), dtype=torch.float32, device=device)


# ----------------------------------------------------------------------------------------------
# raw calls
# ----------------------------------------------------------------------------------------------
_uniform_scale: Dict[Tuple, torch.Tensor] = {}


def row_scale(mask: Optional[torch.Tensor], Bq: int, Nq: int, device) -> torch.Tensor:
    lib = _lib.load()
    device = torch.device(device)
    if mask is None:
        # 1/Nq for every row (model.py:391): a constant of the shape — computed once, not once per step
        key = (device.index, Bq, Nq)
        out = _uniform_scale.get(key)
        if out is None:
            out = torch.empty(Bq * Nq, dtype=torch.float32, device=device)
            with torch.cuda.device(device):
                check(lib.triad_row_scale(None, Bq, Nq, out.data_ptr(), _stream(device)), "triad_row_scale")
                torch.cuda.current_stream(device).synchronize()      # read-only from here on, from any stream
            if len(_uniform_scale) > 64:
                _uniform_scale.clear()
            _uniform_scale[key] = out
        return out
    _require_cuda(mask)
    out = torch.empty(Bq * Nq, dtype=torch.float32, device=device)
    mask = mask.to(torch.int64).contiguous()
    if mask.shape != (Bq, Nq):
        raise ValueError(f"attention_mask must be ({Bq},{Nq}), got {tuple(mask.shape)}")
    with torch.cuda.device(device):
        check(lib.triad_row_scale(_ptr(mask), Bq, Nq, out.data_ptr(), _stream(device)), "triad_row_scale")
    return out


def idx_dtype(Nv: int) -> torch.dtype:
    return torch.uint8 if Nv <= 256 else torch.uint16


def nq_padded(Nq: int) -> int:
    """Row pitch of one query inside the argmax index buffer ([Bv][Bq][nq_pad], see include/triad_b200.h)."""
    return (Nq + 15) // 16 * 16


def idx_buffer(Bv: int, Bq: int, Nq: int, Nv: int, device) -> torch.Tensor:
    """Argmax index buffer [Bv, Bq*nq_padded(Nq)] for a forward.  The kernels never write the entries a >= Nq of a
    query's run (the padding up to nq_pad); they are set to 0 here so that the whole buffer is defined, and two
    forwards of the same inputs give equal buffers whatever memory they were allocated from."""
    nqp = nq_padded(Nq)
    idx = torch.empty(Bv, Bq * nqp, dtype=idx_dtype(Nv), device=device)
    if nqp != Nq:
        idx.view(Bv, Bq, nqp)[:, :, Nq:].zero_()
    return idx


def idx_to_reference_layout(idx: torch.Tensor, Bq: int, Nq: int) -> torch.Tensor:
    """Library layout [Bv, Bq*nq_pad] -> the reference's torch.max(token_sims, dim=3)[1]: (Bq,Bv,Nq) int64."""
    Bv = idx.shape[0]
    return idx.view(Bv, Bq, nq_padded(Nq))[:, :, :Nq].permute(1, 0, 2).to(torch.int64).contiguous()


def maxmean_fwd(q: torch.Tensor, v: torch.Tensor, scale: torch.Tensor, T: torch.Tensor,
                want_idx: bool = True, flags: int = 0, check_watchdog: bool = False):
    """clip fp32 [Bq,Bv], idx [Bv, Bq*nq_padded(Nq)] (uint8/uint16) or None."""
    lib = _lib.load()
    _require_cuda(q, v, scale, T)
    if q.dtype != v.dtype:
        raise TypeError("q and v must have the same dtype")
    q, v = q.contiguous(), v.contiguous()
    Bq, Nq, D = q.shape
    Bv, Nv, D2 = v.shape
    if D != D2:
        raise ValueError("embedding dims differ")
    dt = _dtype_code(q)
    clip = torch.empty(Bq, Bv, dtype=torch.float32, device=q.device)
    idx = idx_buffer(Bv, Bq, Nq, Nv, q.device) if want_idx else None
    nws = lib.triad_maxmean_fwd_workspace_bytes_ex(Bq, Bv, Nq, Nv, D, dt, int(flags))
    with _on(q):
        ws = _Workspace.get(nws, q.device, "fwd")
        st = _stream(q.device)
        check(lib.triad_maxmean_fwd(q.data_ptr(), v.data_ptr(), scale.data_ptr(), T.data_ptr(),
                                    Bq, Bv, Nq, Nv, D, dt, clip.data_ptr(), _ptr(idx),
                                    ws.data_ptr(), ws.numel(), flags, st), "triad_maxmean_fwd")
        if check_watchdog:
            check(lib.triad_maxmean_fwd_status(ws.data_ptr(), st), "triad_maxmean_fwd (watchdog)")
    return clip, idx


def _check_out(t: torch.Tensor, shape, dtype, name: str) -> None:
    if t.dtype != dtype or tuple(t.shape) != tuple(shape) or not t.is_contiguous() or t.device.type != "cuda":
        raise ValueError(f"{name} must be a contiguous {dtype} CUDA tensor of shape {tuple(shape)}")


def maxmean_fwd_nonneg(q: torch.Tensor, v: torch.Tensor, scale: torch.Tensor, T: torch.Tensor, lo: float, coef: float,
                       flags: int = 0, idx: Optional[torch.Tensor] = None, N: Optional[torch.Tensor] = None,
                       sums: Optional[torch.Tensor] = None):
    """The max-mean forward AND N = dL/d<q,v> of the dense non-negative-pressure regulariser (coef * T * clamp'(S) * S
    for every token pair, bf16 [Bq*Nq, Bv*Nv]) from one pass over the similarities (triad_maxmean_fwd_nonneg).
    Returns clip fp32 [Bq,Bv], idx, N, sums fp64 [2] = {sum clamp(S,lo,0)^2, sum dS*<q,v>}.

    A caller that sweeps the images in chunks passes its own outputs: `idx` ([Bv, Bq*nq_padded(Nq)], e.g. the chunk's
    rows of a whole-batch index buffer), `N` (a row-major [Bq*Nq, >= Bv*Nv] bf16 buffer reused across chunks: the
    first Bv*Nv columns are written, the row pitch is N.stride(0)) and `sums` (fp64 [2], ADDED to)."""
    lib = _lib.load()
    _require_cuda(q, v, scale, T)
    if q.dtype != torch.bfloat16 or v.dtype != torch.bfloat16:
        raise TypeError("maxmean_fwd_nonneg takes bfloat16 embeddings")
    q, v = q.contiguous(), v.contiguous()
    Bq, Nq, D = q.shape
    Bv, Nv, D2 = v.shape
    if D != D2:
        raise ValueError("embedding dims differ")
    clip = torch.empty(Bq, Bv, dtype=torch.float32, device=q.device)
    if idx is None:
        idx = idx_buffer(Bv, Bq, Nq, Nv, q.device)
    _check_out(idx, (Bv, Bq * nq_padded(Nq)), idx_dtype(Nv), "idx")
    if N is None:
        N = torch.empty(Bq * Nq, Bv * Nv, dtype=torch.bfloat16, device=q.device)
    if (N.dtype != torch.bfloat16 or N.dim() != 2 or N.shape[0] != Bq * Nq or N.shape[1] < Bv * Nv or N.stride(1) != 1
            or N.device != q.device):
        raise ValueError(f"N must be a row-major bf16 [{Bq * Nq}, >= {Bv * Nv}] tensor on {q.device}")
    if sums is None:
        sums = torch.zeros(2, dtype=torch.float64, device=q.device)
    _check_out(sums, (2,), torch.float64, "sums")
    nws = lib.triad_maxmean_fwd_nonneg_workspace_bytes(Bq, Bv, Nq, Nv, D)
    with _on(q):
        ws = _Workspace.get(nws, q.device, "fwd")
        check(lib.triad_maxmean_fwd_nonneg(q.data_ptr(), v.data_ptr(), scale.data_ptr(), T.data_ptr(), Bq, Bv, Nq, Nv, D,
                                           clip.data_ptr(), idx.data_ptr(), float(lo), float(coef), N.data_ptr(), N.stride(0),
                                           sums.data_ptr(), ws.data_ptr(), ws.numel(), int(flags), _stream(q.device)),
              "triad_maxmean_fwd_nonneg")
    return clip, idx, N, sums


def dense_grad_gemm(N: torch.Tensor, x: torch.Tensor, mode: int) -> torch.Tensor:
    """mode 0: N @ x (N [M,Kc] bf16, x [Kc,D]); mode 1: N.t() @ x (x [M,D]) — the dense regulariser's two backward GEMMs
    on the tensor cores (triad_dense_grad_gemm: MN-major operands, no transposed copies).  bf16 out."""
    lib = _lib.load()
    _require_cuda(N, x)
    if N.dtype != torch.bfloat16 or x.dtype != torch.bfloat16 or N.dim() != 2 or x.dim() != 2:
        raise TypeError("dense_grad_gemm takes 2-D bfloat16 matrices")
    if N.stride(1) != 1:
        raise ValueError("N must be row-major")
    x = x.contiguous()
    M, Kc = N.shape
    D = x.shape[1]
    if x.shape[0] != (Kc if mode == 0 else M):
        raise ValueError("dense_grad_gemm: inner dimensions differ")
    out = torch.empty(M if mode == 0 else Kc, D, dtype=torch.bfloat16, device=N.device)
    nws = lib.triad_dense_grad_gemm_workspace_bytes(M, Kc, D, int(mode))
    with _on(N):
        ws = _Workspace.get(nws, N.device, "dgemm")
        check(lib.triad_dense_grad_gemm(N.data_ptr(), N.stride(0), M, Kc, x.data_ptr(), D, int(mode), out.data_ptr(),
                                        ws.data_ptr(), ws.numel(), _stream(N.device)), "triad_dense_grad_gemm")
    return out


def dense_grad_gemm_f32(N: torch.Tensor, x: torch.Tensor, mode: int, out: torch.Tensor, accumulate: bool) -> torch.Tensor:
    """dense_grad_gemm with an fp32 result written into `out` ([M, D] for mode 0, [Kc, D] for mode 1, contiguous —
    a row slice of a larger buffer will do), or added to it when `accumulate` (triad_dense_grad_gemm_f32)."""
    lib = _lib.load()
    _require_cuda(N, x, out)
    if N.dtype != torch.bfloat16 or x.dtype != torch.bfloat16 or N.dim() != 2 or x.dim() != 2:
        raise TypeError("dense_grad_gemm_f32 takes 2-D bfloat16 matrices")
    if N.stride(1) != 1:
        raise ValueError("N must be row-major")
    x = x.contiguous()
    M, Kc = N.shape
    D = x.shape[1]
    if x.shape[0] != (Kc if mode == 0 else M):
        raise ValueError("dense_grad_gemm_f32: inner dimensions differ")
    _check_out(out, (M if mode == 0 else Kc, D), torch.float32, "out")
    nws = lib.triad_dense_grad_gemm_workspace_bytes(M, Kc, D, int(mode))
    with _on(N):
        ws = _Workspace.get(nws, N.device, "dgemm")
        check(lib.triad_dense_grad_gemm_f32(N.data_ptr(), N.stride(0), M, Kc, x.data_ptr(), D, int(mode), out.data_ptr(),
                                            1 if accumulate else 0, ws.data_ptr(), ws.numel(), _stream(N.device)),
              "triad_dense_grad_gemm_f32")
    return out


def maxmean_bwd(q, v, idx, g, clip, scale, T, need_dq=True, need_dv=True, need_dT=True, dv_f32=False,
                flags: int = 0, dv_out: Optional[torch.Tensor] = None):
    """dv_out: write dv there (fp32 [Bv,Nv,D]) instead of a new tensor; with flags BWD_ACCUMULATE_DV it is added to."""
    lib = _lib.load()
    q, v, g = q.contiguous(), v.contiguous(), g.contiguous()
    if g.dtype != torch.float32:
        g = g.float()
    Bq, Nq, D = q.shape
    Bv, Nv, _ = v.shape
    dt = _dtype_code(q)
    dq = torch.empty_like(q) if need_dq else None
    if dv_out is not None:
        _check_out(dv_out, (Bv, Nv, D), torch.float32, "dv_out")
        need_dv, dv_f32 = True, True
    dv = dv_out if dv_out is not None else (
        torch.empty(Bv, Nv, D, dtype=torch.float32 if dv_f32 else v.dtype, device=v.device) if need_dv else None)
    dT = torch.empty((), dtype=torch.float32, device=q.device) if need_dT else None
    nws = lib.triad_maxmean_bwd_workspace_bytes(Bq, Bv, Nq, Nv, D, dt)
    with _on(q):
        ws = _Workspace.get(nws, q.device, "bwd")
        check(lib.triad_maxmean_bwd(q.data_ptr(), v.data_ptr(), idx.data_ptr(), g.data_ptr(), _ptr(clip),
                                    scale.data_ptr(), T.data_ptr(), Bq, Bv, Nq, Nv, D, dt,
                                    _ptr(dq), _ptr(dv), 1 if dv_f32 else 0, _ptr(dT),
                                    ws.data_ptr(), ws.numel(), int(flags), _stream(q.device)), "triad_maxmean_bwd")
    return dq, dv, dT


def infonce_partial(clip_rows: torch.Tensor, B: int, row0: int):
    lib = _lib.load()
    rows = clip_rows.shape[0]
    row_lse = torch.empty(rows, dtype=torch.float32, device=clip_rows.device)
    col_part = torch.empty(2, B, dtype=torch.float32, device=clip_rows.device)
    nws = lib.triad_infonce_workspace_bytes(rows, B)
    with _on(clip_rows):
        ws = _Workspace.get(nws, clip_rows.device, "nce")
        check(lib.triad_infonce_partial(clip_rows.data_ptr(), rows, B, row0, row_lse.data_ptr(), col_part.data_ptr(),
                                        ws.data_ptr(), ws.numel(), _stream(clip_rows.device)), "triad_infonce_partial")
    return row_lse, col_part


def infonce_finish(clip_rows, B, row0, row_lse, col_parts, grad_scale: float = 1.0):
    lib = _lib.load()
    rows = clip_rows.shape[0]
    col_parts = col_parts.contiguous()
    nparts = col_parts.numel() // (2 * B)
    g = torch.empty(rows, B, dtype=torch.float32, device=clip_rows.device)
    sums = torch.empty(8, dtype=torch.float64, device=clip_rows.device)
    nws = lib.triad_infonce_workspace_bytes(rows, B)
    with _on(clip_rows):
        ws = _Workspace.get(nws, clip_rows.device, "nce")
        check(lib.triad_infonce_finish(clip_rows.data_ptr(), rows, B, row0, row_lse.data_ptr(), col_parts.data_ptr(),
                                       nparts, grad_scale, g.data_ptr(), sums.data_ptr(),
                                       ws.data_ptr(), ws.numel(), _stream(clip_rows.device)), "triad_infonce_finish")
    return g, sums


HEAD_MAX_B = 2048      # triad_contrastive_head: 64 row blocks of 32


def contrastive_head(clip: torch.Tensor, T: Optional[torch.Tensor]):
    """Fused single-device head: g fp32 [B,B], sums fp64 [8], out fp32 [4] = (contrastive, l_cal, sum, d l_cal/dT)."""
    lib = _lib.load()
    B = clip.shape[0]
    g = torch.empty(B, B, dtype=torch.float32, device=clip.device)
    sums = torch.empty(8, dtype=torch.float64, device=clip.device)
    out = torch.empty(4, dtype=torch.float32, device=clip.device)
    nws = lib.triad_contrastive_head_workspace_bytes(B)
    with _on(clip):
        ws = _Workspace.get(nws, clip.device, "head")
        check(lib.triad_contrastive_head(clip.data_ptr(), B, _ptr(T), g.data_ptr(), sums.data_ptr(), out.data_ptr(),
                                         ws.data_ptr(), ws.numel(), _stream(clip.device)), "triad_contrastive_head")
    return g, sums, out


# ----------------------------------------------------------------------------------------------
# autograd
# ----------------------------------------------------------------------------------------------
class MaxMeanSimilarity(torch.autograd.Function):
    """clip[i,j] = sum_a scale[i,a] * max_p round(T <q[i,a], v[j,p]>); backward through the saved
    argmax (src/model.py:387-391 and its autograd backward)."""

    @staticmethod
    def forward(ctx, q, v, temperature, scale, flags, uniform_scale=False, nonneg_lo=None, bwd_pack=False):
        """nonneg_lo: also produce N = dL/d<q,v> of mean(clamp(S, nonneg_lo, 0)^2) over all token pairs and its sums in
        the same pass (returned as non-differentiable extras for regularizers.DenseNonNegFromN); else they are None."""
        T = temperature_tensor(temperature, q.device)
        N = sums = None
        if nonneg_lo is None:
            clip, idx = maxmean_fwd(q, v, scale, T, want_idx=True, flags=flags)
        else:
            numel = float(q.shape[0] * q.shape[1]) * v.shape[0] * v.shape[1]
            clip, idx, N, sums = maxmean_fwd_nonneg(q, v, scale, T, nonneg_lo, 2.0 / numel, flags=flags)
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(q, v, T, scale, idx, clip)
        # rows dropped in the forward (zero weight) have no winners recorded: the backward must skip them too (and may
        # skip zero-weight rows in any case: bwd_pack)
        ctx.bwd_flags = _lib.BWD_PACK_ROWS if ((flags & _lib.FWD_PACK_ROWS) or bwd_pack) else 0
        if uniform_scale:                       # no attention mask: every row has weight 1/Nq, the dv sort need not look
            ctx.bwd_flags |= _lib.BWD_UNIFORM_SCALE
        ctx.mark_non_differentiable(idx)
        if N is not None:
            ctx.mark_non_differentiable(N, sums)
        ctx.t_shape = temperature.shape if isinstance(temperature, torch.Tensor) else None
        ctx.t_dtype = temperature.dtype if isinstance(temperature, torch.Tensor) else None
        return clip, idx, N, sums

    @staticmethod
    def backward(ctx, g, _gidx, _gN=None, _gsums=None):
        q, v, T, scale, idx, clip = ctx.saved_tensors
        if g is None:
            return None, None, None, None, None, None, None, None
        need_dq, need_dv, need_dT = ctx.needs_input_grad[0], ctx.needs_input_grad[1], ctx.needs_input_grad[2]
        dq, dv, dT = maxmean_bwd(q, v, idx, g, clip, scale, T, need_dq, need_dv, need_dT, flags=ctx.bwd_flags)
        if dT is not None and ctx.t_shape is not None:
            dT = dT.reshape(ctx.t_shape).to(ctx.t_dtype)
        return dq, dv, dT, None, None, None, None, None


class SymmetricInfoNCE(torch.autograd.Function):
    """loss = mean_i(-log_softmax_row(clip)[i,i] - log_softmax_col(clip)[i,i]) / 2
    (src/model.py:453-459); forward also produces dLoss/dclip and the statistics sums."""

    @staticmethod
    def forward(ctx, clip):
        clip = clip.contiguous()
        if clip.dtype != torch.float32:
            clip = clip.float()
        B = clip.shape[0]
        if clip.shape[1] != B:
            raise ValueError("InfoNCE needs a square clip-similarity matrix")
        row_lse, col_part = infonce_partial(clip, B, 0)
        g, sums = infonce_finish(clip, B, 0, row_lse, col_part.reshape(1, 2, B))
        loss = (sums[0] / (2 * B)).to(torch.float32)
        ctx.save_for_backward(g)
        ctx.mark_non_differentiable(sums)
        return loss, sums

    @staticmethod
    def backward(ctx, gl, _gs):
        (g,) = ctx.saved_tensors
        return g * gl


class ContrastiveHead(torch.autograd.Function):
    """(contrastive, l_cal, contrastive + l_cal, sums) from the fp32 clip matrix and the temperature parameter:
    symmetric InfoNCE (src/model.py:453-459 / :572-578), its statistics sums and the temperature-calibration term
    20*relu(-log T)^2 (model.py:420-427) in two launches (triad_contrastive_head).  `temperature` may be None
    (no calibration term: the text-visual loss, model.py:544-593, has none)."""

    @staticmethod
    def forward(ctx, clip, temperature):
        clip = clip.contiguous()
        if clip.dtype != torch.float32:
            clip = clip.float()
        B = clip.shape[0]
        if clip.dim() != 2 or clip.shape[1] != B:
            raise ValueError("InfoNCE needs a square clip-similarity matrix")
        T = temperature_tensor(temperature, clip.device) if temperature is not None else None
        g, sums, out = contrastive_head(clip, T)
        ctx.set_materialize_grads(False)          # unused outputs arrive as None, not as zero tensors to add
        ctx.save_for_backward(g, out)
        ctx.t_meta = (temperature.shape, temperature.dtype) if isinstance(temperature, torch.Tensor) else None
        ctx.mark_non_differentiable(sums)
        return out[0], out[1], out[2], sums

    @staticmethod
    def backward(ctx, g_con, g_cal, g_tot, _gs):
        g, out = ctx.saved_tensors
        up = g_con if g_tot is None else (g_tot if g_con is None else g_con + g_tot)
        dclip = g * up if (up is not None and ctx.needs_input_grad[0]) else None
        dT = None
        if ctx.t_meta is not None and ctx.needs_input_grad[1]:
            upc = g_cal if g_tot is None else (g_tot if g_cal is None else g_cal + g_tot)
            if upc is not None:
                dT = (out[3] * upc).reshape(ctx.t_meta[0]).to(ctx.t_meta[1])
        return dclip, dT
