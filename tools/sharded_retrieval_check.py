#!/usr/bin/env python
"""torchrun helper (>= 2 ranks, NCCL): gallery-sharded top-k (triad_b200.dist.sharded_retrieve_topk) against the
single-GPU top-k over the whole gallery — ids bit-equal on every rank, uneven shards, ties across shards.
With --fp8 the gallery is an e4m3 Fp8Gallery and each rank scores its slice of it.  With --ragged it is a
RaggedGallery of captions with cfg 3's lengths; each rank builds its shard from its own caption range, and both
directions are checked (with --fp8 too, an e4m3 RaggedGallery)."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402


def main():
    world, rank, local = int(os.environ["WORLD_SIZE"]), int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    from triad_b200 import retrieval as R
    from triad_b200.dist import sharded_retrieve_topk
    fp8 = "--fp8" in sys.argv[1:]
    ok = True
    if "--ragged" in sys.argv[1:]:
        ok = check_ragged(world, rank, dev, fp8)
    for n_img, Nv, Nq, k in (() if "--ragged" in sys.argv[1:] else ((1001, 256, 77, 10), (515, 1024, 250, 20), (3, 64, 5, 8))):
        g = torch.Generator(device=dev).manual_seed(17)                 # same gallery on every rank
        q = torch.nn.functional.normalize(torch.randn(Nq, 512, generator=g, device=dev), dim=1).bfloat16()
        gal = torch.nn.functional.normalize(torch.randn(n_img, Nv, 512, generator=g, device=dev), dim=2).bfloat16()
        gal[n_img - 1] = gal[0]                                         # a tie across the first and the last shard
        base, rem = n_img // world, n_img % world
        n_loc = base + (1 if rank < rem else 0)
        id0 = rank * base + min(rank, rem)
        if fp8:
            gal = R.quantize_gallery(gal)
            shard = gal[id0:id0 + n_loc]                                # a view: per-patch scales make slices exact
        else:
            shard = gal[id0:id0 + n_loc].contiguous()
        s, ids = sharded_retrieve_topk(q, shard, 1.5, k, id0)
        kk = min(k, n_img)
        s0, i0 = R.retrieve_topk(q, gal, 1.5, kk)
        good = torch.equal(ids[:kk], i0.to(torch.int64)) and torch.equal(s[:kk], s0)
        print(f"rank {rank}: {'fp8 ' if fp8 else ''}n_img={n_img} Nv={Nv} Nq={Nq} k={k}: ids equal {good}", flush=True)
        ok &= good
    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0 and flag.item() == 1:
        print("SHARDED_RETRIEVAL_OK", flush=True)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if flag.item() == 1 else 1)


def check_ragged(world, rank, dev, fp8=False):
    import numpy as np
    from triad_b200 import retrieval as R
    from triad_b200.dist import sharded_retrieve_topk
    ok = True
    for n_cap, Nq, k in ((2001, 256, 10), (777, 1024, 20), (3, 5, 8)):
        g = torch.Generator(device=dev).manual_seed(19)                 # same captions on every rank
        lens = np.random.default_rng(n_cap).integers(8, 78, size=n_cap)
        q = torch.nn.functional.normalize(torch.randn(Nq, 512, generator=g, device=dev), dim=1).bfloat16()
        flat = torch.nn.functional.normalize(torch.randn(int(lens.sum()), 512, generator=g, device=dev), dim=1).bfloat16()
        caps = list(torch.split(flat, [int(x) for x in lens]))
        caps[n_cap - 1] = caps[0]                                       # a tie across the first and the last shard
        base, rem = n_cap // world, n_cap % world
        n_loc = base + (1 if rank < rem else 0)
        id0 = rank * base + min(rank, rem)
        shard = R.RaggedGallery.from_list(caps[id0:id0 + n_loc], fp8=fp8)
        whole = R.RaggedGallery.from_list(caps, fp8=fp8)
        for d in (0, 1):
            s, ids = sharded_retrieve_topk(q, shard, 1.5, k, id0, direction=d)
            kk = min(k, n_cap)
            s0, i0 = R.retrieve_topk(q, whole, 1.5, kk, d)
            good = torch.equal(ids[:kk], i0.to(torch.int64)) and torch.equal(s[:kk], s0)
            print(f"rank {rank}: {'fp8 ' if fp8 else ''}ragged n_cap={n_cap} Nq={Nq} k={k} direction {d}: ids equal {good}", flush=True)
            ok &= good
    return ok


if __name__ == "__main__":
    main()
