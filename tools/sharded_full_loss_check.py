#!/usr/bin/env python
"""torchrun helper (NCCL): the row-sharded full loss (triad_b200.dist.sharded_full_loss_step) against the single-GPU
drop-in full loss (compute_all_similarities_* + compute_contrastive_loss_* + backward, merged forward) on the gathered
batch — every rank compares its loss terms, clip rows, dq / dv shards and temperature gradients — and, on rank 0, a
small shape against fp64 autograd of the oracle's full loss.  Prints SHARDED_FULL_LOSS_OK when every rank passes."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402


def rel(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return ((a - b).norm() / b.norm().clamp(min=1e-30)).item()


def inputs(kind, B, Nq, Nv, D, dev, seed):
    """The same whole batch on every rank."""
    g = torch.Generator(device=dev).manual_seed(seed)
    q = (torch.randn(B, Nq, D, generator=g, device=dev) * 2 / D ** 0.5).bfloat16()
    v = (torch.randn(B, Nv, D, generator=g, device=dev) * 2 / D ** 0.5).bfloat16()
    mask = None
    if kind == "tv":
        lens = torch.randint(8, Nq + 1, (B,), generator=g, device=dev)
        lens[0] = Nq
        mask = (torch.arange(Nq, device=dev)[None, :] < lens[:, None]).to(torch.int64)
    return q, v, mask


def check_vs_dropin(kind, Bl, Nq, Nv, D, world, rank, dev):
    import triad_b200
    from triad_b200.dist import sharded_full_loss_step
    B = Bl * world
    T, thr, w = 0.8, 0.01, 0.5
    q, v, mask = inputs(kind, B, Nq, Nv, D, dev, 29)
    m = triad_b200.TriadHotPath(T, thr, w).to(dev)
    qd, vd = q.clone().requires_grad_(), v.clone().requires_grad_()
    if kind == "av":
        clip, tok = m.compute_all_similarities_av(qd, vd)
        total = m.compute_contrastive_loss_av(clip, tok)[0]
    else:
        clip, tok = m.compute_all_similarities_tv(qd, vd, mask)
        total = m.compute_contrastive_loss_tv(clip, tok)[0]
    clip32 = tok.clip.detach().clone()
    total.backward()
    sl = slice(rank * Bl, (rank + 1) * Bl)
    out = sharded_full_loss_step(q[sl].contiguous(), v[sl].contiguous(), torch.tensor(T, device=dev), kind,
                                 None if mask is None else mask[sl].contiguous(),
                                 patch_sparsity_threshold=thr, patch_sparsity_weight=w)
    dT_sum = out["dT"].clone()
    dist.all_reduce(dT_sum)
    errs = {"total": abs(out["total"].item() - total.item()) / abs(total.item()),
            "clip": rel(out["clip_rows"], clip32[sl]),
            "dq": rel(out["dq"], qd.grad[sl]), "dv": rel(out["dv"], vd.grad[sl]),
            "dT_global": abs(out["dT_global"].item() - m.temperature.grad.item()) / abs(m.temperature.grad.item()),
            "dT_shares": abs(dT_sum.item() - m.temperature.grad.item()) / abs(m.temperature.grad.item())}
    ok = (errs["total"] < 1e-5 and errs["clip"] < 1e-6 and errs["dq"] < 4e-3 and errs["dv"] < 4e-3
          and errs["dT_global"] < 1e-4 and errs["dT_shares"] < 1e-4)
    print(f"rank {rank}: {kind} B={B} {Nq}x{Nv} D={D} vs the single-GPU drop-in: "
          + " ".join(f"{k} {e:.2e}" for k, e in errs.items()) + f" -> {ok}", flush=True)
    return ok


def check_vs_oracle(kind, Bl, Nq, Nv, D, world, rank, dev):
    """Every rank runs its shard; rank 0 gathers dq / dv and compares with fp64 autograd of the full loss."""
    from oracle import oracle as O
    from triad_b200.dist import sharded_full_loss_step
    B = Bl * world
    T, thr, w = 0.8, 0.01, 0.5
    q, v, mask = inputs(kind, B, Nq, Nv, D, dev, 31)
    sl = slice(rank * Bl, (rank + 1) * Bl)
    out = sharded_full_loss_step(q[sl].contiguous(), v[sl].contiguous(), torch.tensor(T, device=dev), kind,
                                 None if mask is None else mask[sl].contiguous(),
                                 patch_sparsity_threshold=thr, patch_sparsity_weight=w)
    dq = torch.empty((world,) + tuple(out["dq"].shape), dtype=out["dq"].dtype, device=dev)
    dv = torch.empty((world,) + tuple(out["dv"].shape), dtype=out["dv"].dtype, device=dev)
    dist.all_gather_into_tensor(dq.view(-1), out["dq"].contiguous().view(-1))
    dist.all_gather_into_tensor(dv.view(-1), out["dv"].contiguous().view(-1))
    if rank != 0:
        return True
    q64, v64 = q.cpu().double().requires_grad_(), v.cpu().double().requires_grad_()
    T64 = torch.tensor(T, dtype=torch.float64, requires_grad=True)
    tok = torch.einsum("iad,jpd->ijap", q64, v64) * T64
    best = tok.max(dim=3).values
    if mask is None:
        clip = best.mean(dim=2)
    else:
        mk = mask.cpu().double()[:, None, :]
        clip = (best * mk).sum(dim=2) / mk.sum(dim=2).clamp(min=1e-7)
    tgt = torch.arange(B)
    con = (-torch.log_softmax(clip, dim=1)[tgt, tgt] - torch.log_softmax(clip.t(), dim=1)[tgt, tgt]).mean() / 2
    reg = O.regularization_av(tok, T64)[0] if kind == "av" else O.regularization_tv(tok, thr, w)
    total = con + reg
    total.backward()
    errs = {"total": abs(out["total"].item() - total.item()) / abs(total.item()),
            "dq": rel(dq.reshape(q.shape).cpu(), q64.grad), "dv": rel(dv.reshape(v.shape).cpu(), v64.grad),
            "dT_global": abs(out["dT_global"].item() - T64.grad.item()) / abs(T64.grad.item())}
    # bf16 inputs against fp64 arithmetic: the similarities are rounded to bf16 as the reference rounds them
    ok = errs["total"] < 1e-3 and errs["dq"] < 2e-2 and errs["dv"] < 2e-2 and errs["dT_global"] < 2e-2
    print(f"rank 0: {kind} B={B} {Nq}x{Nv} D={D} vs the fp64 oracle: "
          + " ".join(f"{k} {e:.2e}" for k, e in errs.items()) + f" -> {ok}", flush=True)
    return ok


def main():
    world, rank, local = int(os.environ["WORLD_SIZE"]), int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    ok = True
    ok &= check_vs_dropin("av", 64, 250, 256, 512, world, rank, dev)
    ok &= check_vs_dropin("tv", 48, 77, 256, 512, world, rank, dev)
    ok &= check_vs_oracle("tv", 3, 12, 24, 64, world, rank, dev)
    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0 and flag.item() == 1:
        print("SHARDED_FULL_LOSS_OK", flush=True)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if flag.item() == 1 else 1)


if __name__ == "__main__":
    main()
