"""Row-sharded contrastive step across the GPUs of one node (SURVEY.md §8(e)).

The reference is single-GPU.  The B x B clip matrix shards naturally by rows: rank r owns
queries and images [r*Bl,(r+1)*Bl).  One exchange each way:

  forward   all-gather(V)                     -> every rank scores its queries against ALL images
            all-gather(column (max,sumexp))   -> 2*B floats per rank, completes the column softmax
            all-gather(8 fp64 sums)           -> loss and the similarity statistics
  backward  reduce(dV partial, fp32), one destination rank at a time, pipelined with the dV gather of the next
            rank's images and with dQ  -> each rank receives the gradient of its own images
            (dQ is local; dT is a sum of the per-rank  sum g*clip  already in the 8 sums)

There is no other data-path collective; per-rank work is (B/W) x B pairs.  sharded_full_loss_step() (autograd face:
sharded_full_loss) is the reference's FULL loss — InfoNCE plus the regularisers — from one pass over the similarities
per image chunk and one fp32 dv reduction per destination rank; sharded_regularizer_step() is the regularisers alone
(one more reduce-scatter of a dv partial).  Collectives go through
torch.distributed (NCCL over NVLink/NVSwitch on the GPU box; gloo in the CPU tests, where the
kernel entry points are injected by the test — the product binding below is CUDA-only).
"""
from __future__ import annotations

from typing import Dict, Optional

import torch
import torch.distributed as dist


class CudaKernels:
    """The product binding: the C-ABI ops."""

    #: set by row_scale(): a mask was given, so zero-weight rows are packed out of the bf16 forward / dq
    packed = False

    def row_scale(self, mask, Bq, Nq, device):
        from . import ops
        self.packed = mask is not None
        return ops.row_scale(mask, Bq, Nq, device)

    def maxmean_fwd(self, q, v, scale, T):
        from . import _lib, ops
        flags = _lib.FWD_PACK_ROWS if (self.packed and q.dtype == torch.bfloat16) else 0
        return ops.maxmean_fwd(q, v, scale, T, want_idx=True, flags=flags)

    def infonce_partial(self, clip_rows, B, row0):
        from . import ops
        return ops.infonce_partial(clip_rows, B, row0)

    def infonce_finish(self, clip_rows, B, row0, row_lse, col_parts):
        from . import ops
        return ops.infonce_finish(clip_rows, B, row0, row_lse, col_parts)

    def maxmean_bwd(self, q, v, idx, g, clip, scale, T):
        from . import ops
        from . import _lib
        flags = _lib.BWD_PACK_ROWS if (self.packed and q.dtype == torch.bfloat16) else 0
        if not self.packed:
            flags |= _lib.BWD_UNIFORM_SCALE
        dq, dv, _ = ops.maxmean_bwd(q, v, idx, g, clip, scale, T, need_dq=True, need_dv=True,
                                    need_dT=False, dv_f32=True, flags=flags)
        return dq, dv


    # dv / dq separately: lets the sharded step reduce one destination rank's dv while the next one is computed
    def maxmean_bwd_dv(self, q, v, idx, g, scale, T):
        from . import ops
        from . import _lib
        _, dv, _ = ops.maxmean_bwd(q, v, idx, g, None, scale, T, need_dq=False, need_dv=True, need_dT=False, dv_f32=True,
                                   flags=0 if self.packed else _lib.BWD_UNIFORM_SCALE)
        return dv

    def maxmean_bwd_dq(self, q, v, idx, g, scale, T):
        from . import _lib, ops
        flags = _lib.BWD_PACK_ROWS if (self.packed and q.dtype == torch.bfloat16) else 0
        dq, _, _ = ops.maxmean_bwd(q, v, idx, g, None, scale, T, need_dq=True, need_dv=False, need_dT=False, flags=flags)
        return dq


    def nonneg(self, q, v, T, lo, numel):
        """Dense non-negative-pressure term of this rank's rows against ALL images, normalised by the global pair
        count: (sum clamp^2 fp64 scalar, dq (Bq,Nq,D), dv partial (Bv,Nv,D) fp32, dT fp64 scalar)."""
        from . import regularizers as R
        sums, dq, dv = R.nonneg_sweep(q, v, T, lo, numel, True, R.CHUNK_BYTES)
        return sums[0], dq.view(q.shape).to(q.dtype), dv.float(), sums[1]

    def pospair(self, q, v, T, kind, threshold):
        """Positive-pair term of this rank's pairs (mean over ITS pairs): temporal smoothness ("av") or patch-usage
        sparsity ("tv").  Returns (value fp64 scalar, dq (Bl,Nq,D), dv (Bl,Nv,D), dT fp64 scalar), unweighted."""
        from . import regularizers as R
        qd, vd = q.detach().requires_grad_(True), v.detach().requires_grad_(True)
        Td = T.detach().clone().requires_grad_(True)
        with torch.enable_grad():                      # also inside an autograd Function's forward (ShardedFullLoss)
            term = R.temporal_smoothness(qd, vd, Td) if kind == "av" else R.patch_sparsity(qd, vd, Td, threshold)
            term.backward()
        return term.detach().double(), qd.grad, vd.grad, Td.grad.double()

    # ---- sharded_full_loss_step: one pass per image chunk, gradients carried in fp32 up to one dv reduction ----
    def full_loss_merged(self, q, v):
        """Shapes the merged forward takes without padding (a zero patch would join the max over patches)."""
        from . import regularizers as R
        return q.dtype == v.dtype and R.fused_supported(q, v) and v.shape[1] % 8 == 0

    def n_buffer(self, rows, cols, device):
        return torch.empty(rows, cols, dtype=torch.bfloat16, device=device)

    def maxmean_fwd_nonneg(self, q, vc, scale, T, lo, coef, idx, N, sums):
        """clip (Bq, jc) of q against the images vc; idx (the chunk's image-major rows) and N = dL/d<q,v> (the first
        jc*Nv columns of the buffer N) written, sums (fp64 [2]) added to."""
        from . import ops
        clip, _, _, _ = ops.maxmean_fwd_nonneg(q, vc, scale, T, lo, coef, idx=idx, N=N, sums=sums)
        return clip

    def dense_grad_f32(self, N, x, mode, out, accumulate):
        """mode 0: out (+)= N x;  mode 1: out (+)= N^T x — fp32, deterministic."""
        from . import ops
        ops.dense_grad_gemm_f32(N, x, mode, out, accumulate)

    def maxmean_bwd_dv_add(self, q, v, idx, g, scale, T, dv):
        """dv (fp32 (Bv,Nv,D)) += the max-mean backward's dv."""
        from . import _lib, ops
        flags = _lib.BWD_ACCUMULATE_DV | (0 if self.packed else _lib.BWD_UNIFORM_SCALE)
        ops.maxmean_bwd(q, v, idx, g, None, scale, T, need_dq=False, need_dv=True, need_dT=False, flags=flags, dv_out=dv)

    def scale(self, x, s):
        """x * s for a 0-dim device scalar s, without a host sync."""
        from . import regularizers as R
        return R.scale_by(x, s)


def _all_gather(x: torch.Tensor, W: int, group) -> torch.Tensor:
    """all-gather along a new leading dim ([W, *x.shape]); flat views keep every backend happy."""
    x = x.contiguous()
    out = torch.empty((W,) + tuple(x.shape), dtype=x.dtype, device=x.device)
    dist.all_gather_into_tensor(out.view(-1), x.view(-1), group=group)
    return out


def _reduce_scatter_rows(x: torch.Tensor, W: int, r: int, group) -> torch.Tensor:
    """sum over ranks of x ([W*n, ...]), returning this rank's n rows.  NCCL: one reduce-scatter
    over NVLink; gloo (CPU tests) has no reduce-scatter, so all-reduce and slice."""
    n = x.shape[0] // W
    if dist.get_backend(group) == "gloo":
        y = x.contiguous().clone()
        dist.all_reduce(y, op=dist.ReduceOp.SUM, group=group)
        return y[r * n:(r + 1) * n].contiguous()
    out = torch.empty((n,) + tuple(x.shape[1:]), dtype=x.dtype, device=x.device)
    dist.reduce_scatter_tensor(out.view(-1), x.contiguous().view(-1), op=dist.ReduceOp.SUM, group=group)
    return out


def combine_all_sums(all_sums: torch.Tensor) -> torch.Tensor:
    """The per-rank fp64 sums ([W,8]) as the sums of the whole batch, on the device: everything adds except the
    hardest negative (index 5), which is a max."""
    s = all_sums.sum(dim=0)
    s[5] = all_sums[:, 5].max()
    return s


def stats_from_all_sums(all_sums: torch.Tensor, B: int, prefix: str) -> Dict[str, float]:
    """Combine the per-rank fp64 sums ([W,8]) into the reference's six statistics (model.py:435-450)."""
    from .model import _stats_from_sums
    return _stats_from_sums(combine_all_sums(all_sums), B, prefix)


def sharded_contrastive_step(q_local: torch.Tensor, v_local: torch.Tensor, temperature: torch.Tensor,
                             mask_local: Optional[torch.Tensor] = None, group=None, kernels=None,
                             need_grads: bool = True) -> Dict[str, torch.Tensor]:
    """One forward(+backward) of max-mean similarity + symmetric InfoNCE over a row-sharded batch.

    q_local (Bl,Nq,D), v_local (Bl,Nv,D): this rank's queries and images.  Returns
    {loss (global, fp32 scalar), all_sums [W,8] fp64, clip_rows (Bl,B), dq (Bl,Nq,D), dv (Bl,Nv,D),
     dT, dT_global (fp32 scalars)} — dq / dv: gradients of the GLOBAL loss w.r.t. this rank's shards; dT: this
    rank's SHARE of the global temperature gradient (the shares add up to dT_global), consistent with what
    back-propagating dq / dv through replicated encoder weights yields on each rank: reduce all of them the
    same way (SUM, or DDP's mean)."""
    k = kernels if kernels is not None else CudaKernels()
    W = dist.get_world_size(group) if dist.is_initialized() else 1
    r = dist.get_rank(group) if dist.is_initialized() else 0
    Bl, Nq, D = q_local.shape
    Nv = v_local.shape[1]
    B = Bl * W
    dev = q_local.device
    q_local, v_local = q_local.contiguous(), v_local.contiguous()
    T = temperature.detach().to(device=dev, dtype=torch.float32).reshape(())

    v_all = _all_gather(v_local, W, group).view(B, Nv, D) if W > 1 else v_local

    scale = k.row_scale(mask_local, Bl, Nq, dev)
    clip_rows, idx = k.maxmean_fwd(q_local, v_all, scale, T)             # (Bl,B), [B, Bl*Nq]
    row_lse, col_part = k.infonce_partial(clip_rows, B, r * Bl)          # (Bl,), (2,B)
    col_parts = _all_gather(col_part, W, group) if W > 1 else col_part.reshape(1, 2, B)
    g, sums = k.infonce_finish(clip_rows, B, r * Bl, row_lse, col_parts)  # (Bl,B), (8,) fp64
    all_sums = _all_gather(sums, W, group) if W > 1 else sums.reshape(1, 8)
    loss = (all_sums[:, 0].sum() / (2 * B)).to(torch.float32)
    out = {"loss": loss, "all_sums": all_sums, "clip_rows": clip_rows, "B": B}
    if not need_grads:
        return out

    if W > 1 and hasattr(k, "maxmean_bwd_dv"):
        # Pipelined: the fp32 dv partial of ONE destination rank's images at a time; its reduction to that rank
        # travels (NCCL's stream) while the next rank's images are gathered for, and dq — which needs no
        # communication — runs under the last reductions.  Same sums as one reduce-scatter of the whole partial.
        works, dv32 = [], None
        for d in range(W):
            sl = slice(d * Bl, (d + 1) * Bl)
            part = k.maxmean_bwd_dv(q_local, v_all[sl], idx[sl], g[:, sl].contiguous(), scale, T)   # (Bl,Nv,D) fp32
            dst = dist.get_global_rank(group, d) if group is not None else d
            works.append(dist.reduce(part, dst=dst, op=dist.ReduceOp.SUM, group=group, async_op=True))
            if d == r:
                dv32 = part
        dq = k.maxmean_bwd_dq(q_local, v_all, idx, g, scale, T)
        for w in works:
            w.wait()
    else:
        dq, dv_partial = k.maxmean_bwd(q_local, v_all, idx, g, clip_rows, scale, T)   # dv_partial (B,Nv,D) fp32
        dv32 = _reduce_scatter_rows(dv_partial, W, r, group) if W > 1 else dv_partial
    out["dq"] = dq
    out["dv"] = dv32.to(v_local.dtype)
    # The temperature is REPLICATED across ranks, so — like the gradient of any replicated parameter reached
    # through dq / dv — each rank returns its own share: sum_{i in this rank's rows, j} g[i,j]*clip[i,j] / T.  A SUM
    # over ranks (or DDP's mean, which scales every replicated parameter by the same 1/W) gives the global gradient.
    out["dT"] = (sums[6] / T.double()).to(torch.float32)
    out["dT_global"] = (all_sums[:, 6].sum() / T.double()).to(torch.float32)
    return out


def sharded_regularizer_step(q_local: torch.Tensor, v_local: torch.Tensor, temperature: torch.Tensor, kind: str,
                             group=None, kernels=None, patch_sparsity_threshold: float = 0.3,
                             patch_sparsity_weight: float = 0.1) -> Dict[str, torch.Tensor]:
    """The reference's regularisation terms (model.py:394-428 for kind "av", :516-542 for "tv") over a row-sharded
    batch, with the gradients of the GLOBAL regulariser w.r.t. this rank's shards:

      dense non-negative pressure   this rank's rows against all (all-gathered) images; value all-reduced, dq local,
                                    the dv partial reduce-scattered like the contrastive one;
      positive-pair terms           (temporal smoothness / patch sparsity on token_sims[i,i]) are local — a rank owns
                                    both members of its positive pairs (triad_pospair_terms);
      temperature calibration       a scalar on T ("av" only).

    Returns {reg, smooth (0.01*l_smooth, "av"), dq (Bl,Nq,D), dv (Bl,Nv,D), dT (this rank's share), dT_global}."""
    from . import regularizers as R
    if kind not in ("av", "tv"):
        raise ValueError("kind must be 'av' or 'tv'")
    k = kernels if kernels is not None else CudaKernels()
    W = dist.get_world_size(group) if dist.is_initialized() else 1
    r = dist.get_rank(group) if dist.is_initialized() else 0
    Bl, Nq, D = q_local.shape
    Nv = v_local.shape[1]
    B = Bl * W
    dev = q_local.device
    q_local, v_local = q_local.detach().contiguous(), v_local.detach().contiguous()
    T = temperature.detach().to(device=dev, dtype=torch.float32).reshape(())
    v_all = _all_gather(v_local, W, group).view(B, Nv, D) if W > 1 else v_local

    lo = -60.0 if kind == "av" else -20.0
    numel = float(B) * B * Nq * Nv
    s2, dq_nn, dv_nn_partial, dT_nn = k.nonneg(q_local, v_all, T, lo, numel)
    dv_nn = _reduce_scatter_rows(dv_nn_partial, W, r, group) if W > 1 else dv_nn_partial

    # positive pairs: local (a rank owns both members of its pairs); the global mean is the mean of the per-rank means
    # (equal shard sizes).  A single token row has no temporal differences: the term is dropped (the reference's mean
    # over an empty tensor would be NaN).
    w_term = 0.01 if kind == "av" else patch_sparsity_weight
    if kind == "av" and Nq <= 1:
        term, dq_pp, dv_pp, dT_pp = (torch.zeros((), dtype=torch.float64, device=dev), torch.zeros_like(q_local),
                                     torch.zeros_like(v_local), torch.zeros((), dtype=torch.float64, device=dev))
    else:
        term, dq_pp, dv_pp, dT_pp = k.pospair(q_local, v_local, T, kind, patch_sparsity_threshold)
    # values are global (all-reduced); the temperature gradient stays this rank's SHARE (see sharded_contrastive_step)
    dT = 0.15 * dT_nn.double() + (w_term / W) * dT_pp.double()
    scal = torch.stack([s2.double() / numel, term.double() / W, dT])
    if W > 1:
        dist.all_reduce(scal, op=dist.ReduceOp.SUM, group=group)
    l_nonneg, l_term, dT_global = scal[0], scal[1], scal[2]
    reg = 0.15 * l_nonneg + w_term * l_term
    if kind == "av":                                   # 20 * relu(-log T)^2 (model.py:414-424): a term on T alone
        Td = T.double()
        neg_log = torch.clamp(-torch.log(Td), min=0)
        reg = reg + 20.0 * neg_log ** 2
        dT = dT - 40.0 * neg_log / Td / W              # every rank carries 1/W of it, so the shares still add up
        dT_global = dT_global - 40.0 * neg_log / Td
    out = {"reg": reg.to(torch.float32), "dT": dT.to(torch.float32), "dT_global": dT_global.to(torch.float32),
           "dq": (0.15 * dq_nn.float() + (w_term / W) * dq_pp.float()).to(q_local.dtype),
           "dv": (0.15 * dv_nn.float() + (w_term / W) * dv_pp.float()).to(v_local.dtype)}
    if kind == "av":
        out["smooth"] = (0.01 * l_term).to(torch.float32)
    return out


def sharded_full_loss_step(q_local: torch.Tensor, v_local: torch.Tensor, temperature: torch.Tensor, kind: str,
                           mask_local: Optional[torch.Tensor] = None, group=None, kernels=None,
                           patch_sparsity_threshold: float = 0.3, patch_sparsity_weight: float = 0.1,
                           chunk_bytes: Optional[int] = None) -> Dict[str, torch.Tensor]:
    """The reference's FULL loss over a row-sharded batch — symmetric InfoNCE of the max-mean similarities plus the
    regularisers (model.py:394-472 for kind "av", :516-593 for "tv") — with its gradients, from ONE pass over the
    similarities:

      forward   all-gather(V); per image chunk (at most `chunk_bytes` of N, default regularizers.chunk_budget) the
                merged tcgen05 pass gives this rank's clip rows, the argmax AND the dense regulariser's N = dL/d<q,v>,
                and two GEMMs turn N into dQ (fp32, accumulated over the chunks) and the chunk's rows of this rank's
                fp32 dV partial;  InfoNCE as in sharded_contrastive_step, the regulariser sums riding on its all-gather
      backward  per destination rank d: the contrastive dv of d's images is ADDED onto the dense dV partial of those
                images (fp32) and the sum goes to d in one reduce; dq (local) runs under the last reductions;
                the positive-pair terms are local (a rank owns both members of its pairs).

    Masked text runs unpacked here, as in the single-GPU merged mode (padded tokens take part in the regulariser,
    model.py:525; their rows carry no contrastive gradient).  Shapes the merged pass does not take (fp32, patch counts
    that are not a multiple of 8, Nv > 256, D > 512) compose sharded_contrastive_step and sharded_regularizer_step.

    Returns {total, contrastive, reg, smooth ("av": 0.01*l_smooth), all_sums [W,8] fp64, clip_rows (Bl,B), dq (Bl,Nq,D),
    dv (Bl,Nv,D), dT, dT_global}: dq / dv are gradients of the GLOBAL total w.r.t. this rank's shards, dT this rank's
    share of the temperature gradient (see sharded_contrastive_step)."""
    from . import ops
    from . import regularizers as R
    if kind not in ("av", "tv"):
        raise ValueError("kind must be 'av' or 'tv'")
    k = kernels if kernels is not None else CudaKernels()
    q_local, v_local = q_local.detach().contiguous(), v_local.detach().contiguous()
    if not k.full_loss_merged(q_local, v_local):
        return _composed_full_loss_step(q_local, v_local, temperature, kind, mask_local, group, k,
                                        patch_sparsity_threshold, patch_sparsity_weight)
    W = dist.get_world_size(group) if dist.is_initialized() else 1
    r = dist.get_rank(group) if dist.is_initialized() else 0
    Bl, Nq, D = q_local.shape
    Nv = v_local.shape[1]
    B, M = Bl * W, Bl * Nq
    dev = q_local.device
    T = temperature.detach().to(device=dev, dtype=torch.float32).reshape(())
    v_all = _all_gather(v_local, W, group).view(B, Nv, D) if W > 1 else v_local
    scale = k.row_scale(mask_local, Bl, Nq, dev)

    # ---- forward: clip rows, argmax and N of the dense term from one pass per image chunk; N -> dQ, dV at once ----
    lo = -60.0 if kind == "av" else -20.0
    numel = float(B) * B * Nq * Nv
    coef = 0.15 * 2.0 / numel                  # N, dQ, dV and sums[1] carry the term's weight
    budget = R.chunk_budget(dev, R.CHUNK_BYTES if chunk_bytes is None else chunk_bytes)
    jc = max(1, min(B, budget // (M * Nv * 2)))
    N = k.n_buffer(M, jc * Nv, dev)            # one buffer, row pitch jc*Nv, reused by every chunk
    clip_rows = torch.empty(Bl, B, dtype=torch.float32, device=dev)
    idx = ops.idx_buffer(B, Bl, Nq, Nv, dev)
    nsums = torch.zeros(2, dtype=torch.float64, device=dev)
    dq_dense = torch.empty(M, D, dtype=torch.float32, device=dev)
    dv_part = torch.empty(B * Nv, D, dtype=torch.float32, device=dev)    # this rank's rows against every image
    q2 = q_local.view(M, D)
    for j0 in range(0, B, jc):
        j1 = min(B, j0 + jc)
        vc = v_all[j0:j1]
        clip_rows[:, j0:j1] = k.maxmean_fwd_nonneg(q_local, vc, scale, T, lo, coef, idx[j0:j1], N, nsums)
        Nc = N[:, :(j1 - j0) * Nv]
        k.dense_grad_f32(Nc, vc.reshape(-1, D), 0, dq_dense, j0 > 0)
        k.dense_grad_f32(Nc, q2, 1, dv_part[j0 * Nv:j1 * Nv], False)
    del N

    # positive pairs: local; the global mean is the mean of the per-rank means (equal shard sizes).  A single token
    # row has no temporal differences: the term is dropped (the reference's mean over an empty tensor would be NaN).
    w_term = 0.01 if kind == "av" else patch_sparsity_weight
    if kind == "av" and Nq <= 1:
        term, dq_pp, dv_pp, dT_pp = (torch.zeros((), dtype=torch.float64, device=dev), torch.zeros_like(q_local),
                                     torch.zeros_like(v_local), torch.zeros((), dtype=torch.float64, device=dev))
    else:
        term, dq_pp, dv_pp, dT_pp = k.pospair(q_local, v_local, T, kind, patch_sparsity_threshold)

    # ---- InfoNCE; the regulariser's per-rank scalars travel with the 8 sums (one all-gather) ----
    row_lse, col_part = k.infonce_partial(clip_rows, B, r * Bl)
    col_parts = _all_gather(col_part, W, group) if W > 1 else col_part.reshape(1, 2, B)
    g, sums = k.infonce_finish(clip_rows, B, r * Bl, row_lse, col_parts)
    dT_reg = nsums[1] + (w_term / W) * dT_pp.double()
    ext = torch.cat([sums.double().reshape(8), torch.stack([nsums[0], term.double().reshape(()), dT_reg])])
    all_ext = _all_gather(ext, W, group) if W > 1 else ext.reshape(1, 11)
    all_sums = all_ext[:, :8].contiguous()
    reg_sums = all_ext[:, 8:].sum(dim=0)
    Td = T.double()
    contrastive = all_sums[:, 0].sum() / (2 * B)
    l_term = reg_sums[1] / W
    reg = 0.15 * reg_sums[0] / numel + w_term * l_term
    dT = sums[6].double() / Td + dT_reg
    dT_global = all_sums[:, 6].sum() / Td + reg_sums[2]
    if kind == "av":                                   # 20 * relu(-log T)^2 (model.py:414-424): a term on T alone
        neg_log = torch.clamp(-torch.log(Td), min=0)
        reg = reg + 20.0 * neg_log ** 2
        dT = dT - 40.0 * neg_log / Td / W              # every rank carries 1/W of it, so the shares still add up
        dT_global = dT_global - 40.0 * neg_log / Td

    # ---- backward: contrastive dv onto the dense dV partial of each destination rank's images, one fp32 reduce ----
    dv_part = dv_part.view(B, Nv, D)
    works = []
    for d in range(W):
        sl = slice(d * Bl, (d + 1) * Bl)
        k.maxmean_bwd_dv_add(q_local, v_all[sl], idx[sl], g[:, sl].contiguous(), scale, T, dv_part[sl])
        if W > 1:
            dst = dist.get_global_rank(group, d) if group is not None else d
            works.append(dist.reduce(dv_part[sl], dst=dst, op=dist.ReduceOp.SUM, group=group, async_op=True))
    dq_con = k.maxmean_bwd_dq(q_local, v_all, idx, g, scale, T)
    for w in works:
        w.wait()
    dq = dq_dense.view(Bl, Nq, D) + dq_con.float() + (w_term / W) * dq_pp.float()
    dv = dv_part[r * Bl:(r + 1) * Bl] + (w_term / W) * dv_pp.float()
    out = {"total": (contrastive + reg).to(torch.float32), "contrastive": contrastive.to(torch.float32),
           "reg": reg.to(torch.float32), "all_sums": all_sums, "clip_rows": clip_rows,
           "dq": dq.to(q_local.dtype), "dv": dv.to(v_local.dtype),
           "dT": dT.to(torch.float32), "dT_global": dT_global.to(torch.float32)}
    if kind == "av":
        out["smooth"] = (0.01 * l_term).to(torch.float32)
    return out


def _composed_full_loss_step(q_local, v_local, temperature, kind, mask_local, group, k, patch_sparsity_threshold,
                             patch_sparsity_weight):
    """sharded_full_loss_step for the shapes the merged pass does not take: the two separate calls."""
    con = sharded_contrastive_step(q_local, v_local, temperature, mask_local, group, k)
    reg = sharded_regularizer_step(q_local, v_local, temperature, kind, group, k, patch_sparsity_threshold,
                                   patch_sparsity_weight)
    out = {"total": con["loss"] + reg["reg"], "contrastive": con["loss"], "reg": reg["reg"],
           "all_sums": con["all_sums"], "clip_rows": con["clip_rows"],
           "dq": (con["dq"].float() + reg["dq"].float()).to(q_local.dtype),
           "dv": (con["dv"].float() + reg["dv"].float()).to(v_local.dtype),
           "dT": con["dT"] + reg["dT"], "dT_global": con["dT_global"] + reg["dT_global"]}
    if kind == "av":
        out["smooth"] = reg["smooth"]
    return out


def merge_topk(scores: torch.Tensor, ids: torch.Tensor, k: int):
    """Top-k of candidate (score, global id) pairs under the library's retrieval order: score descending, ties to the
    lower id (retrieve.cu::make_key; a stable argsort of -scores over ids in ascending order, retrieval.py:125)."""
    by_id = torch.argsort(ids, stable=True)
    s, i = scores[by_id], ids[by_id]
    order = torch.argsort(s, descending=True, stable=True)[:k]
    return s[order], i[order]


def sharded_retrieve_topk(q_feats: torch.Tensor, gallery_shard: torch.Tensor, temperature, k: int, id0: int,
                          group=None, direction: int = 0, local_topk=None):
    """BASELINE cfg 5 across GPUs (SURVEY.md §8(e), replaces the gallery loop of retrieval.py:161-175): the gallery is
    sharded BY IMAGES — this rank holds images [id0, id0 + n_local) — every rank scores the (replicated) query against
    its shard and keeps its local top-k, the k (score, global id) pairs of every rank are all-gathered (2*k*W numbers)
    and merged with the single-GPU ordering.  Returns (scores fp32 [k], ids int64 [k]), identical on every rank and
    bit-identical to retrieve_topk over the whole gallery on one GPU.

    `local_topk(q, gallery, temperature, k, direction) -> (scores, local ids)` is the scoring kernel (the CUDA
    retrieve_topk by default; the CPU tests inject an oracle-backed stand-in)."""
    if local_topk is None:
        from .retrieval import retrieve_topk as local_topk
    W = dist.get_world_size(group) if dist.is_initialized() else 1
    n_local = gallery_shard.shape[0]
    kl = min(k, n_local)
    s, ids = local_topk(q_feats, gallery_shard, temperature, kl, direction)
    cand_s = torch.full((k,), float("-inf"), dtype=torch.float32, device=s.device)
    cand_i = torch.full((k,), torch.iinfo(torch.int64).max, dtype=torch.int64, device=s.device)
    cand_s[:kl] = s.float()
    cand_i[:kl] = ids.to(torch.int64) + int(id0)
    if W > 1:
        cand_s = _all_gather(cand_s, W, group).reshape(-1)
        cand_i = _all_gather(cand_i, W, group).reshape(-1)
    return merge_topk(cand_s, cand_i, k)


class ShardedContrastiveLoss(torch.autograd.Function):
    """Autograd face of sharded_contrastive_step: the forward computes the loss AND the gradients
    (the saved argmax indices never outlive the call); backward scales them by the incoming grad.

    Every returned gradient — the temperature's included — is this rank's SHARE of the global one: reduce the
    parameter gradients across ranks with a SUM (or let DDP average all of them alike)."""

    @staticmethod
    def forward(ctx, q_local, v_local, temperature, mask_local, group):
        out = sharded_contrastive_step(q_local, v_local, temperature, mask_local, group)
        ctx.save_for_backward(out["dq"], out["dv"], out["dT"])
        ctx.t_like = temperature
        ctx.mark_non_differentiable(out["all_sums"])
        return out["loss"], out["all_sums"]

    @staticmethod
    def backward(ctx, gl, _gs):
        dq, dv, dT = ctx.saved_tensors
        return dq * gl.to(dq.dtype), dv * gl.to(dv.dtype), (dT * gl).reshape(ctx.t_like.shape).to(ctx.t_like.dtype), None, None


class ShardedFullLoss(torch.autograd.Function):
    """Autograd face of sharded_full_loss_step: the forward computes the loss terms AND the gradients; backward
    scales them by the incoming gradient of `total` (a device scalar: no host sync).  Only `total` is
    differentiable; contrastive / reg / smooth / the combined sums are reported values."""

    @staticmethod
    def forward(ctx, q_local, v_local, temperature, kind, mask_local, group, kernels, options):
        k = kernels if kernels is not None else CudaKernels()
        out = sharded_full_loss_step(q_local, v_local, temperature, kind, mask_local, group, k, **options)
        ctx.save_for_backward(out["dq"], out["dv"], out["dT"])
        ctx.kernels = k
        ctx.t_meta = (temperature.shape, temperature.dtype)
        smooth = out["smooth"] if "smooth" in out else torch.zeros_like(out["reg"])
        sums = combine_all_sums(out["all_sums"])
        ctx.mark_non_differentiable(out["contrastive"], out["reg"], smooth, sums)
        return out["total"], out["contrastive"], out["reg"], smooth, sums

    @staticmethod
    def backward(ctx, g_total, *_):
        dq, dv, dT = ctx.saved_tensors
        k = ctx.kernels
        gT = (dT * g_total).reshape(ctx.t_meta[0]).to(ctx.t_meta[1])
        return k.scale(dq, g_total), k.scale(dv, g_total), gT, None, None, None, None, None


def sharded_full_loss(q_local: torch.Tensor, v_local: torch.Tensor, temperature: torch.Tensor, kind: str,
                      mask_local: Optional[torch.Tensor] = None, group=None, kernels=None,
                      patch_sparsity_threshold: float = 0.3, patch_sparsity_weight: float = 0.1,
                      chunk_bytes: Optional[int] = None):
    """The reference's loss call over a row-sharded batch: (total, contrastive, reg, 0.01*l_smooth, stats) for kind
    "av" (compute_contrastive_loss_av, model.py:430-472), (total, stats) for "tv" (model.py:544-593).  `stats` is the
    reference's statistics dictionary of the WHOLE batch, read from the device on first access.

    Only `total` is differentiable: back-propagating it puts on q_local / v_local the gradients of the global total
    w.r.t. this rank's shards and on `temperature` this rank's share (reduce parameter gradients across ranks with a
    SUM, or let DDP average all of them alike).  The other values are detached reports."""
    opts = {"patch_sparsity_threshold": patch_sparsity_threshold, "patch_sparsity_weight": patch_sparsity_weight,
            "chunk_bytes": chunk_bytes}
    total, contrastive, reg, smooth, sums = ShardedFullLoss.apply(q_local, v_local, temperature, kind, mask_local,
                                                                  group, kernels, opts)
    from .model import LazyStats
    W = dist.get_world_size(group) if dist.is_initialized() else 1
    stats = LazyStats(sums, q_local.shape[0] * W, kind)
    if kind == "av":
        return total, contrastive, reg, smooth, stats
    return total, stats
