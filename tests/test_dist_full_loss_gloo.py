"""CPU tier: the row-sharded full-loss step (triad_b200/dist.py: sharded_full_loss_step, sharded_full_loss) over a
world_size-2 gloo group gives the loss terms, statistics and gradients of fp64 autograd of the reference's FULL loss
(max-mean + symmetric InfoNCE + regularisers, model.py:394-472 / :516-593) on the whole batch.  The kernels are
oracle-backed stand-ins defined here; the C-ABI additions the step uses are checked for argument validation."""
import ctypes
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import oracle as O
from tests.cpu_kernels import PipelinedOracleKernels

B, NQ, NV, D = 6, 9, 20, 16
T_VAL = 0.9                  # < 1: the calibration term is active
THR, W_SPARSE = 0.02, 0.5
CHUNK_BYTES = 2 * (B // 2) * NQ * NV * 2   # bf16 N of 2 images x a 3-query shard: 3 chunks per rank, boundaries inside rank blocks


class FullLossOracleKernels(PipelinedOracleKernels):
    """Stand-ins of the entry points sharded_full_loss_step adds: the merged chunk forward (the max-mean oracle plus
    fp64 N = dL/d<q,v> of the clamp term), the fp32 gradient GEMMs with and without accumulation, the accumulating
    dv backward, the device-scalar scale."""

    def full_loss_merged(self, q, v):
        return True

    def n_buffer(self, rows, cols, device):
        return torch.full((rows, cols), float("nan"), dtype=torch.float64)

    def maxmean_fwd_nonneg(self, q, vc, scale, T, lo, coef, idx, N, sums):
        clip, lib_idx = self.maxmean_fwd(q, vc, scale, T)
        idx.copy_(lib_idx.to(idx.dtype))
        Bq, Nq, Dm = q.shape
        raw = q.double().reshape(-1, Dm) @ vc.double().reshape(-1, Dm).t()
        S = float(T) * raw
        c = S.clamp(min=lo, max=0)
        n = coef * c * (S >= lo).double() * float(T)
        N[:, :n.shape[1]] = n
        sums[0] += c.pow(2).sum()
        sums[1] += (n * raw).sum() / float(T)
        return clip

    def dense_grad_f32(self, N, x, mode, out, accumulate):
        r = (N @ x.double()) if mode == 0 else (N.t() @ x.double())
        if accumulate:
            out.add_(r.float())
        else:
            out.copy_(r.float())

    def maxmean_bwd_dv_add(self, q, v, idx, g, scale, T, dv):
        dv.add_(self.maxmean_bwd_dv(q, v, idx, g, scale, T))

    def scale(self, x, s):
        return x * s.to(x.dtype)

    def pospair(self, q, v, T, kind, threshold):
        with torch.enable_grad():
            return super().pospair(q, v, T, kind, threshold)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _inputs(kind):
    q, v, mask = O.make_inputs(B, NQ, NV, D, torch.float32, seed=11, masked=(kind == "tv"))
    return q * 3, v * 3, mask                # some similarities below zero by a margin


def _reference(kind):
    """fp64 autograd of the full loss on the whole batch: dense token tensor, max-mean, symmetric InfoNCE, the
    oracle's restatement of the regularisers."""
    q, v, mask = _inputs(kind)
    q64, v64 = q.double().requires_grad_(), v.double().requires_grad_()
    T64 = torch.tensor(T_VAL, dtype=torch.float64, requires_grad=True)
    tok = torch.einsum("iad,jpd->ijap", q64, v64) * T64
    best = tok.max(dim=3).values
    if mask is None:
        clip = best.mean(dim=2)
    else:
        m = mask.double()[:, None, :]
        clip = (best * m).sum(dim=2) / m.sum(dim=2).clamp(min=1e-7)
    tgt = torch.arange(B)
    con = (-torch.log_softmax(clip, dim=1)[tgt, tgt] - torch.log_softmax(clip.t(), dim=1)[tgt, tgt]).mean() / 2
    if kind == "av":
        reg, smooth = O.regularization_av(tok, T64)
    else:
        reg, smooth = O.regularization_tv(tok, THR, W_SPARSE), None
    total = con + reg
    total.backward()
    return {"total": total.item(), "contrastive": con.item(), "reg": reg.item(),
            "smooth": None if smooth is None else smooth.item(), "clip": clip.detach(),
            "dq": q64.grad, "dv": v64.grad, "dT": T64.grad.item()}


def _run(kind, rank, world):
    from triad_b200.dist import sharded_full_loss_step, stats_from_all_sums
    q, v, mask = _inputs(kind)
    Bl = B // world
    sl = slice(rank * Bl, (rank + 1) * Bl)
    out = sharded_full_loss_step(q[sl], v[sl], torch.tensor(T_VAL), kind, mask[sl] if mask is not None else None,
                                 kernels=FullLossOracleKernels(), patch_sparsity_threshold=THR,
                                 patch_sparsity_weight=W_SPARSE, chunk_bytes=CHUNK_BYTES)
    res = {key: (val.item() if val.dim() == 0 else val) for key, val in out.items()}
    res["stats"] = stats_from_all_sums(out["all_sums"], B, kind)
    return res


def _worker(rank, world, port, kind, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        ret[rank] = _run(kind, rank, world)
    finally:
        dist.destroy_process_group()


def _check_rank(o, ref, kind, rank, Bl):
    sl = slice(rank * Bl, (rank + 1) * Bl)
    for key in ("total", "contrastive", "reg") + (("smooth",) if kind == "av" else ()):
        assert abs(o[key] - ref[key]) < 1e-5 * abs(ref[key]), (key, o[key], ref[key])
    assert abs(o["dT_global"] - ref["dT"]) < 1e-4 * abs(ref["dT"])
    assert torch.allclose(o["dq"].double(), ref["dq"][sl], rtol=1e-4, atol=1e-7)
    assert torch.allclose(o["dv"].double(), ref["dv"][sl], rtol=1e-4, atol=1e-7)
    assert torch.allclose(o["clip_rows"].double(), ref["clip"][sl], rtol=1e-5, atol=1e-6)
    for key, val in O.similarity_stats(ref["clip"], kind).items():
        assert abs(o["stats"][key] - val) < 1e-5, key


def test_chunk_plan_splits_rank_blocks():
    """The forced budget gives 3 chunks of 2 images over the 6 images: the boundary at image 2 falls inside rank 0's
    block [0, 3) and the one at 4 inside rank 1's block [3, 6)."""
    Bl = B // 2
    jc = CHUNK_BYTES // (Bl * NQ * NV * 2)
    assert jc == 2 and (B + jc - 1) // jc >= 3
    assert any(0 < j0 < Bl for j0 in range(0, B, jc)) and any(Bl < j0 < B for j0 in range(0, B, jc))


@pytest.mark.parametrize("kind", ["av", "tv"])
def test_two_rank_full_loss_matches_full_batch(kind):
    world = 2
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), kind, ret), nprocs=world, join=True)
    ref = _reference(kind)
    for r in range(world):
        _check_rank(ret[r], ref, kind, r, B // world)
    # the temperature is replicated: the per-rank shares add up to the global gradient
    assert abs(sum(ret[r]["dT"] for r in range(world)) - ref["dT"]) < 1e-4 * abs(ref["dT"])


@pytest.mark.parametrize("kind", ["av", "tv"])
def test_single_process_full_loss(kind):
    ref = _reference(kind)
    o = _run(kind, 0, 1)
    _check_rank(o, ref, kind, 0, B)
    assert abs(o["dT"] - ref["dT"]) < 1e-4 * abs(ref["dT"])


def test_autograd_face_scales_and_accumulates():
    """backward of 2.5*total gives exactly 2.5x the eager gradients; a phase-weighted av + tv sum accumulates both
    on the shared image embeddings and the temperature."""
    from triad_b200.dist import sharded_full_loss, sharded_full_loss_step
    k = FullLossOracleKernels()
    opts = dict(kernels=k, patch_sparsity_threshold=THR, patch_sparsity_weight=W_SPARSE, chunk_bytes=CHUNK_BYTES)
    qa, v, _ = _inputs("av")
    qt, _, mask = _inputs("tv")
    T = torch.tensor(T_VAL)
    eager_av = sharded_full_loss_step(qa, v, T, "av", **opts)
    eager_tv = sharded_full_loss_step(qt, v, T, "tv", mask, **opts)

    qa_p, v_p, T_p = qa.clone().requires_grad_(), v.clone().requires_grad_(), T.clone().requires_grad_()
    total, con, reg, smooth, stats = sharded_full_loss(qa_p, v_p, T_p, "av", **opts)
    assert total.requires_grad and not con.requires_grad and not reg.requires_grad and not smooth.requires_grad
    assert abs(total.item() - eager_av["total"].item()) == 0.0
    assert abs(stats["av_hardest_negative"] - O.similarity_stats(eager_av["clip_rows"], "av")["av_hardest_negative"]) < 1e-6
    (2.5 * total).backward()
    assert torch.equal(qa_p.grad, eager_av["dq"] * 2.5)
    assert torch.equal(v_p.grad, eager_av["dv"] * 2.5)
    assert torch.equal(T_p.grad, (eager_av["dT"] * 2.5).reshape(()))

    qa_p.grad = v_p.grad = T_p.grad = None
    qt_p = qt.clone().requires_grad_()
    tot_av = sharded_full_loss(qa_p, v_p, T_p, "av", **opts)[0]
    tot_tv, stats_tv = sharded_full_loss(qt_p, v_p, T_p, "tv", mask, **opts)
    assert "tv_separation" in stats_tv
    (0.7 * tot_av + 0.3 * tot_tv).backward()
    assert torch.allclose(v_p.grad, eager_av["dv"] * 0.7 + eager_tv["dv"] * 0.3, rtol=1e-6, atol=1e-9)
    assert torch.allclose(qa_p.grad, eager_av["dq"] * 0.7, rtol=1e-6, atol=0)
    assert torch.allclose(qt_p.grad, eager_tv["dq"] * 0.3, rtol=1e-6, atol=0)
    assert torch.allclose(T_p.grad, (eager_av["dT"] * 0.7 + eager_tv["dT"] * 0.3).reshape(()), rtol=1e-6)


def test_library_additions_validate_arguments_without_gpu():
    """triad_dense_grad_gemm_f32 and TRIAD_BWD_ACCUMULATE_DV reject bad arguments before any CUDA call."""
    from triad_b200 import _lib, build
    build.build()
    lib = _lib.load()
    ARG, ALIGN, WS = -1, -3, -4
    null = None
    one = ctypes.c_void_p(16)
    odd = ctypes.c_void_p(24)
    f = lib.triad_dense_grad_gemm_f32
    ws = lib.triad_dense_grad_gemm_workspace_bytes(256, 512, 64, 0)
    assert ws == lib.triad_dense_grad_gemm_workspace_bytes(256, 512, 64, 0) > 256
    assert f(null, 512, 256, 512, one, 64, 0, one, 0, one, ws, null) == ARG       # N
    assert f(one, 512, 256, 512, null, 64, 0, one, 0, one, ws, null) == ARG       # x
    assert f(one, 512, 256, 512, one, 64, 0, null, 1, one, ws, null) == ARG       # out
    assert f(one, 512, 256, 512, one, 64, 0, one, 0, null, ws, null) == ARG       # ws
    assert f(one, 512, 256, 512, one, 64, 2, one, 0, one, ws, null) == ARG        # mode
    assert f(one, 512, 256, 512, one, 64, 0, one, 2, one, ws, null) == ARG        # accumulate is 0 or 1
    assert f(one, 512, 256, 512, one, 64, 0, odd, 1, one, ws, null) == ALIGN
    b = lib.triad_maxmean_bwd
    acc = _lib.BWD_ACCUMULATE_DV
    assert acc == 1024
    # bf16 inputs with a bf16 dv: nothing to accumulate into in fp32
    assert b(one, one, one, one, one, one, one, 2, 2, 4, 8, 64, 1, one, one, 0, one, one, 1 << 20, acc, null) == ARG
    # fp32 dv (dv_f32 = 1, or fp32 inputs): accepted, the call goes on to the workspace check
    assert b(one, one, one, one, one, one, one, 2, 2, 4, 8, 64, 1, one, one, 1, one, one, 256, acc, null) == WS
    assert b(one, one, one, one, one, one, one, 2, 2, 4, 8, 64, 0, one, one, 0, one, one, 256, acc, null) == WS
    for bad in (512, 512 | acc, 2048):
        assert b(one, one, one, one, one, one, one, 2, 2, 4, 8, 64, 1, one, one, 1, one, one, 256, bad, null) == ARG, bad
