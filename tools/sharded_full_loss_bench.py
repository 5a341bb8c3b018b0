#!/usr/bin/env python
"""Times the row-sharded FULL loss step (contrastive + regularisers) two ways on the same inputs:

  one_pass  triad_b200.dist.sharded_full_loss_step: one merged pass over the similarities per image chunk, one fp32
            dv reduction per destination rank
  composed  sharded_contrastive_step + sharded_regularizer_step: the contrastive sweep, then the regulariser-only sweep
            and a second dv reduction

Both arms compute the loss and every gradient.  They run in the same process, alternated (A B A B ...), every shape
warmed up first; each step is timed with CUDA events.  Shapes: one rank at cfg 2 (av, B=256, 250 x 256) and cfg 3 (tv,
B=512, 77 masked text tokens); under torchrun with >= 2 ranks the cfg 4 rank shape (B=8192 over the ranks).

    python tools/sharded_full_loss_bench.py [--steps 10] [--warmup 3]
    torchrun --nproc-per-node=8 tools/sharded_full_loss_bench.py
"""
import argparse
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import bench  # noqa: E402


def device_line(index):
    """Name, power limit and SM clock limit of the card, read next to the numbers they qualify."""
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        if r.returncode == 0 and r.stdout.strip():
            return r.stdout.strip()
    except Exception:
        pass
    return torch.cuda.get_device_name(index) + ", power limit unknown"


def run_shape(cfg_key, world, rank, local, dev, steps, warmup):
    from triad_b200.dist import sharded_contrastive_step, sharded_full_loss_step, sharded_regularizer_step
    cfg = dict(bench.CONFIGS[cfg_key])
    Bl = cfg["B"] // world                            # the global batch, rows sharded over the ranks
    kind = "tv" if cfg["masked"] else "av"
    (q, v, mask), = bench.make_device_inputs(cfg, Bl, 1234 + rank, dev, 1)
    T = torch.tensor(1.5, device=dev)

    def one_pass():
        o = sharded_full_loss_step(q, v, T, kind, mask)
        return o["total"], o["dq"], o["dv"]

    def composed():
        c = sharded_contrastive_step(q, v, T, mask)
        r = sharded_regularizer_step(q, v, T, kind)
        return (c["loss"] + r["reg"], (c["dq"].float() + r["dq"].float()).to(q.dtype),
                (c["dv"].float() + r["dv"].float()).to(v.dtype))

    arms = {"one_pass": one_pass, "composed": composed}
    res = {}
    for name, fn in arms.items():                     # warm-up, and the two arms' results side by side
        for _ in range(warmup):
            res[name] = fn()
    torch.cuda.synchronize()
    agree = {"total_rel": abs(res["one_pass"][0].item() - res["composed"][0].item()) / abs(res["composed"][0].item()),
             "dq_rel": bench.rel_err(res["one_pass"][1].float(), res["composed"][1].float()),
             "dv_rel": bench.rel_err(res["one_pass"][2].float(), res["composed"][2].float())}
    del res
    times = {n: [] for n in arms}
    with bench.ClockSampler(local) as clocks:
        for _ in range(steps):
            for name, fn in arms.items():
                if world > 1:
                    dist.barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                times[name].append(e0.elapsed_time(e1))
    ck = clocks.summary()
    if rank == 0:
        print(f"{cfg['name']}: {world} rank(s), per-rank shape B_local={Bl} of B={Bl * world}, kind {kind}")
        for name in arms:
            t = times[name]
            print(f"  {name:9s} median {statistics.median(t):9.3f} ms/step  min {min(t):9.3f}  max {max(t):9.3f}  "
                  f"({len(t)} steps, alternated)")
        print(f"  one_pass / composed (medians): {statistics.median(times['one_pass']) / statistics.median(times['composed']):.3f}")
        print(f"  agreement one_pass vs composed: total {agree['total_rel']:.2e}  dq {agree['dq_rel']:.2e}  "
              f"dv {agree['dv_rel']:.2e} (relative)")
        print(f"  SM clock during the timed steps: median {ck.get('sm_mhz')} MHz (min {ck.get('sm_mhz_min')}, "
              f"max allowed {ck.get('sm_max_mhz')}), board power max {ck.get('power_w_max')} W, "
              f"clock-event reasons {ck.get('reasons')}", flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("sharded_full_loss_bench needs a CUDA device")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if rank == 0:
        print(f"device: {device_line(local)}  (torch {torch.__version__}, CUDA {torch.version.cuda})", flush=True)
    shapes = ["cfg2", "cfg3"] if world == 1 else ["cfg4"]
    for key in shapes:
        run_shape(key, world, rank, local, dev, args.steps, args.warmup)
        torch.cuda.empty_cache()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
