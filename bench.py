#!/usr/bin/env python
"""Benchmark of the fused max-mean similarity + symmetric InfoNCE path (fwd + bwd).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl triad|reference] [--config auto|cfg2|cfg3|cfg4]
                    [--verify] [--no-extras] [--no-cpu-baseline] [--dump-outputs DIR]

metric: clip-pairs/sec = B_global^2 / t(step)   (BASELINE.json).  One "step" = one forward + backward of the hot path
over one synthetic batch.  N=1 runs BASELINE cfg 2 (B=256, 250 frames x 256 patches, D=512, bf16); N>1 (launched by
torchrun, one rank per GPU) runs cfg 4 (B=8192 global, rows sharded over the ranks, NCCL all-gather / reduce).
Rank 0 prints ONE JSON line.

`value`        device-resident inputs, CUDA-event timing, max over ranks.
`e2e`          the same step through the public drop-in API starting from PINNED HOST buffers (H2D copies of the
               embeddings and the D2H read of the loss inside the timed region).
`roofline`     the tcgen05 forward kernel against the measured bf16 peak (MEASURED_PEAKS.json), plus the whole step.
`cpu_baseline` the reference's own step (oracle/_ref, staged by oracle/build_ref.py; the oracle port if absent) on this
               box's host cores, bounded sample.
N=1 extras (each with its own clock sample and roofline): `full_loss`, `cfg3`, `cfg4_rank_shape_1gpu`, `cfg4_1gpu`
(the B=8192 step on ONE GPU: the strong-scaling denominator of the N>1 lines), `cfg5` (retrieval, HBM-bound).
N>1 extras: `parity` (the W-rank step vs the single-GPU step on the gathered batch, on the GPUs, before timing)
and `cfg5_sharded` (gallery sharded by images, local top-k + all-gather merge).
`--impl reference`: only the CPU arm, as its own JSON line.   `--verify`: only the N-rank parity check.
`--dump-outputs DIR` (N=1): what the last timed step returned to its caller, as DIR/<name>.npy (see dump_outputs).  The
inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CONFIGS = {
    "cfg2": dict(B=256, Nq=250, Nv=256, D=512, masked=False,
                 name="cfg2: B=256, 250 HuBERT frames x 256 DINOv2 patches, D=512, bf16 fwd+bwd"),
    "cfg3": dict(B=512, Nq=77, Nv=256, D=512, masked=True,
                 name="cfg3: B=512, 77 text tokens (ragged masks, n_i in [8,77]) x 256 patches, D=512, bf16 fwd+bwd"),
    "cfg4": dict(B=8192, Nq=250, Nv=256, D=512, masked=False,
                 name="cfg4: B=8192 global, 250 x 256, D=512, bf16 fwd+bwd, rows sharded over ranks"),
}
CFG5 = dict(n_img=100000, Nv=1024, D=512, k=10,
            name="cfg5: 1 query x 100 000 gallery images x 1024 patches, D=512, bf16, forward-only top-10")


def algorithmic_flops(B_cols, n_tokens_total, Nv, D):
    """SURVEY.md §8(d): 2*Bcols*(sum n_i)*Nv*D forward + 4*Bcols*(sum n_i)*D sparse backward."""
    return 2.0 * B_cols * n_tokens_total * Nv * D, 4.0 * B_cols * n_tokens_total * D


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"bf16": float(d["bf16_tflops"]), "bf16_sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                "hbm": float(d["hbm_gbs"]), "source": "measured (MEASURED_PEAKS.json)"}
    return {"bf16": 1590.0, "bf16_sustained": 1400.0, "hbm": 6500.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """SM clock, board power and clock-event (throttle) reasons during a timed region (B200_PROFILING.md's clocks
    line).  Sampled in-process through NVML every 10 ms (tools/sampler_ab.py: no measurable effect on the step);
    `nvidia-smi -lms 25` — whose start-up alone takes ~0.1 s, i.e. misses short regions — is the fallback."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    # nvmlClocksEventReasons bits
    BITS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4),
            ("hw_power_brake", 0x80))

    def __init__(self, index=0):
        self.rows, self.proc, self.index, self.nv, self.stop = [], None, index, None, False

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:
            import torch
            uuid = str(torch.cuda.get_device_properties(self.index).uuid)
            return pynvml, pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
        except Exception:
            return pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.index)

    def _poll(self):
        nv, h = self.nv
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        while not self.stop:
            try:
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                self.rows.append([nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM), mx, nv.nvmlDeviceGetPowerUsage(h) / 1e3]
                                 + ["Active" if r & bit else "Not Active" for _, bit in self.BITS])
            except Exception:
                pass
            time.sleep(0.01)

    def __enter__(self):
        try:
            self.nv = self._nvml_handle()
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            time.sleep(0.02)                    # the first sample is out before the timed region starts
            return self
        except Exception:
            self.nv = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "25"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            time.sleep(0.08)
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *a):
        if self.nv is not None:
            time.sleep(0.02)
            self.stop = True
            self.t.join(timeout=1)
        elif self.proc is not None:
            time.sleep(0.05)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, pw, reasons = [], 0.0, [], set()
        names = [n for n, _ in self.BITS]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1])); pw.append(float(r[2]))
                for n, val in zip(names, r[3:3 + len(names)]):
                    if str(val).lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm),
                "sm_mhz_min": min(sm), "power_w_max": max(pw) if pw else None,
                "source": "nvml" if self.nv is not None else "nvidia-smi"}


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's own step on the host cores
# ------------------------------------------------------------------------------------------------
def cpu_reference_step_factory(cfg, B_sample):
    """Returns (step, kind, what).  kind "reference": the unmodified reference methods from oracle/_ref (staged by
    oracle/build_ref.py): compute_all_similarities_{av,tv} + compute_contrastive_loss_{av,tv} with the regularisers
    bound to zero, i.e. the reference's own similarity / max-mean / statistics / InfoNCE lines and autograd backward —
    the like-for-like of the metric.  kind "port": the oracle's restatement of the same lines, when oracle/_ref is
    not there."""
    import torch
    from oracle import oracle as O
    from oracle import ref_loader
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    q, v, mask = O.make_inputs(B_sample, cfg["Nq"], cfg["Nv"], cfg["D"], torch.float32, seed=1234,
                               masked=cfg["masked"], min_len=8)
    q.requires_grad_(True)
    v.requires_grad_(True)
    ref = ref_loader.load()
    if ref is not None:
        M = ref[0].MultiModalModel
        stub = ref_loader.make_stub(M, 1.5, regularizers=False)

        def step():
            q.grad = v.grad = stub.temperature.grad = None
            if mask is None:
                clip, tok = M.compute_all_similarities_av(stub, q, v)
                total = M.compute_contrastive_loss_av(stub, clip, tok)[0]
            else:
                clip, tok = M.compute_all_similarities_tv(stub, q, v, mask)
                total = M.compute_contrastive_loss_tv(stub, clip, tok)[0]
            total.backward()
            return float(total)
        return step, "reference", ("the reference's own methods, unmodified (oracle/_ref/model.py: compute_all_similarities_* + "
                                   "compute_contrastive_loss_* with zero regularisers), fp32, autograd backward")
    T = torch.tensor(1.5, requires_grad=True)

    def step_port():
        q.grad = v.grad = T.grad = None
        loss, _, _ = O.reference_step_autograd(q, v, T, mask)
        return float(loss)
    return step_port, "port", "oracle.reference_step_autograd (restatement of the reference's materialising fwd+bwd), fp32"


def cpu_baseline(cfg, budget_s=12.0, B_sample=32):
    import torch
    step, kind, what = cpu_reference_step_factory(cfg, B_sample)
    step()                                   # warm-up
    t0, n = time.perf_counter(), 0
    while True:
        step(); n += 1
        el = time.perf_counter() - t0
        if el >= budget_s or n >= 50:
            break
    return {"value": B_sample * B_sample * n / el, "unit": "clip-pairs/s", "cores": torch.get_num_threads(),
            "kind": kind,
            "sample": f"{what}, on a B={B_sample} sub-batch of the same shape (Nq={cfg['Nq']}, Nv={cfg['Nv']}, "
                      f"D={cfg['D']}), {n} steps in {el:.1f} s; pairs/s is per-pair work, so it transfers to the full batch"}


def run_reference(args, cfg_key):
    """--impl reference: the reference's CPU implementation of the path, all host threads, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    cfg = CONFIGS[cfg_key]
    Bs = 32
    step, kind, what = cpu_reference_step_factory(cfg, Bs)
    for _ in range(max(args.warmup, 1)):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    el = time.perf_counter() - t0
    val = Bs * Bs * args.steps / el
    cores = torch.get_num_threads()
    sample = f"each step = fwd+bwd of {what} on a B={Bs} sub-batch of {cfg['name']}"
    print(json.dumps({
        "impl": "reference", "metric": "clip-pairs/sec", "value": val, "unit": "clip-pairs/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfg["name"], "sample_batch": Bs},
        "cpu_baseline": {"value": val, "unit": "clip-pairs/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": "clip-pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def make_device_inputs(cfg, B_local, seed, device, n_sets):
    import torch
    g = torch.Generator(device=device).manual_seed(seed)
    sets = []
    for _ in range(n_sets):
        q = (torch.randn(B_local, cfg["Nq"], cfg["D"], generator=g, device=device) / cfg["D"] ** 0.5).to(torch.bfloat16)
        v = (torch.randn(B_local, cfg["Nv"], cfg["D"], generator=g, device=device) / cfg["D"] ** 0.5).to(torch.bfloat16)
        mask = None
        if cfg["masked"]:
            lens = torch.randint(8, cfg["Nq"] + 1, (B_local,), generator=g, device=device)
            lens[0] = cfg["Nq"]
            mask = (torch.arange(cfg["Nq"], device=device)[None, :] < lens[:, None]).to(torch.int64)
        sets.append((q, v, mask))
    return sets


def rel_err(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return ((a - b).norm() / b.norm().clamp(min=1e-30)).item()


DUMP_ROWS = 32          # batch rows that --dump-outputs writes of the batch-sized outputs


def dump_outputs(path, outs):
    """Writes one step's results as path/<name>.npy, float32: `loss`, `grad_temperature`, and on DUMP_ROWS batch rows
    drawn with a fixed seed (listed in `sample_rows`) `clip_sims` [DUMP_ROWS, B], `grad_q` [DUMP_ROWS, Nq, D] and
    `grad_v` [DUMP_ROWS, Nv, D].  Whole, the two gradients of cfg 2 would take 130 MB each, clip_sims of cfg 4 268 MB."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    B = outs["clip_sims"].shape[0]
    rows = torch.randperm(B, generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort().values
    arrays = {"loss": outs["loss"], "grad_temperature": outs["grad_temperature"], "sample_rows": rows}
    for name in ("clip_sims", "grad_q", "grad_v"):
        arrays[name] = outs[name][rows.to(outs[name].device)]
    for name, t in arrays.items():
        np.save(os.path.join(path, name + ".npy"), t.detach().float().cpu().numpy())


def verify_sharded(world, rank, dev, group=None):
    """N-rank parity on the GPUs (NCCL): sharded_contrastive_step on W shards vs the single-GPU drop-in on the gathered
    batch (every rank recomputes it), unmasked and masked; and, at a small size, vs the CPU oracle on rank 0.
    Returns a dict; raises AssertionError on a mismatch."""
    import torch
    import torch.distributed as dist
    import triad_b200
    from triad_b200.dist import sharded_contrastive_step
    out = {"parity_nranks": world}
    worst = {"loss": 0.0, "dq": 0.0, "dv": 0.0, "dT": 0.0, "clip": 0.0}
    for masked, (Bl, Nq, Nv, D) in ((False, (64, 250, 256, 512)), (True, (48, 77, 256, 512)), (False, (8, 50, 256, 512))):
        B = Bl * world
        cfg = dict(Nq=Nq, Nv=Nv, D=D, masked=masked)
        (q, v, mask), = make_device_inputs(cfg, B, 4242 + Nq, dev, 1)          # same seed on every rank: same full batch
        sl = slice(rank * Bl, (rank + 1) * Bl)
        T = torch.tensor(1.5, device=dev)
        sh = sharded_contrastive_step(q[sl].contiguous(), v[sl].contiguous(), T, None if mask is None else mask[sl].contiguous(),
                                      group=group)
        m = triad_b200.TriadHotPath(temperature=1.5).to(dev)
        m.triad_regularizers = False
        qd, vd = q.clone().requires_grad_(True), v.clone().requires_grad_(True)
        if mask is None:
            clip, tok = m.compute_all_similarities_av(qd, vd)
            con = m.compute_contrastive_loss_av(clip, tok)[1]
        else:
            clip, tok = m.compute_all_similarities_tv(qd, vd, mask)
            con = m.compute_contrastive_loss_tv(clip, tok)[0]
        con.backward()
        dT_sum = sh["dT"].clone()
        if world > 1:
            dist.all_reduce(dT_sum, op=dist.ReduceOp.SUM, group=group)
        errs = {"loss": abs(sh["loss"].item() - con.item()) / abs(con.item()),
                "clip": rel_err(sh["clip_rows"], tok.clip.detach()[sl]),
                "dq": rel_err(sh["dq"], qd.grad[sl]), "dv": rel_err(sh["dv"], vd.grad[sl]),
                "dT": abs(dT_sum.item() - m.temperature.grad.item()) / max(abs(m.temperature.grad.item()), 1e-12),
                "dT_global": abs(sh["dT_global"].item() - m.temperature.grad.item()) / max(abs(m.temperature.grad.item()), 1e-12)}
        # same kernels, same winners: clip rows agree to the fp32 summation order of the per-group partial sums (the
        # 32-row groups start at the shard's first row); g then differs only by that and by the order in which the
        # column partials are combined, so dq / dv agree to well below one bf16 rounding
        assert errs["clip"] < 2e-6, (masked, errs)
        assert errs["loss"] < 1e-6 and errs["dq"] < 2e-3 and errs["dv"] < 2e-3, (masked, errs)
        assert errs["dT"] < 1e-3 and errs["dT_global"] < 1e-3, (masked, errs)
        for k in worst:
            worst[k] = max(worst[k], errs[k])
        if Bl == 8 and rank == 0:               # and the oracle, where it finishes in seconds
            from oracle import oracle as O
            ref = O.contrastive_step_closed_form(q.cpu(), v.cpu(), 1.5, None)
            e = {"loss": abs(sh["loss"].item() - ref["loss"].item()) / abs(ref["loss"].item()),
                 "dq": rel_err(sh["dq"].cpu(), ref["dq"][sl]), "dv": rel_err(sh["dv"].cpu(), ref["dv"][sl])}
            assert e["loss"] < 1e-5 and e["dq"] < 1e-2 and e["dv"] < 1e-2, e
            out["vs_oracle"] = e
    out["parity"] = "ok"
    out["worst_rel_err_vs_single_gpu"] = worst
    return out


def run_triad(args, cfg_key):
    import torch
    import torch.distributed as dist
    import triad_b200
    from triad_b200 import _lib
    from triad_b200.dist import CudaKernels, sharded_contrastive_step

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    _lib.check(lib.triad_device_check(local), "triad_device_check")
    peaks = measured_peaks()

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, K):
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(K):
            fn(i)
        e1.record()
        sync_all()
        ms = torch.tensor([e0.elapsed_time(e1) / K], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    # ---- N-rank parity on the GPUs, before anything is timed -------------------------------------
    parity = None
    if world > 1 or args.verify:
        parity = verify_sharded(world, rank, dev)
        if args.verify:
            if rank == 0:
                print(json.dumps(parity), flush=True)
            if world > 1:
                dist.barrier()
                dist.destroy_process_group()
            return parity

    cfg = CONFIGS[cfg_key]
    B = cfg["B"]
    assert B % world == 0
    Bl = B // world
    n_sets = 3 if world == 1 else 2
    sets = make_device_inputs(cfg, Bl, 1234 + rank, dev, n_sets)
    in_bytes = sum(t.numel() * t.element_size() for t in sets[0][:2])
    model = triad_b200.TriadHotPath(temperature=1.5).to(dev)
    model.triad_regularizers = False       # BASELINE.json's metric: max-mean similarity + InfoNCE, fwd + bwd
    T = model.temperature
    fwd_ev = []
    last_step = {}

    def api_step(m, q, v, mask, record=False):
        """One step through the drop-in methods (the calls forward_audio_visual / forward_text_visual make); its results
        are kept in last_step until the next step."""
        q.grad = v.grad = m.temperature.grad = None
        if record:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        if mask is None:
            clip, tok = m.compute_all_similarities_av(q, v)
        else:
            clip, tok = m.compute_all_similarities_tv(q, v, mask)
        if record:
            e1.record(); fwd_ev.append((e0, e1))
        total = m.compute_contrastive_loss_av(clip, tok)[0] if mask is None else m.compute_contrastive_loss_tv(clip, tok)[0]
        total.backward()
        last_step.update(loss=total, clip_sims=clip, grad_q=q.grad, grad_v=v.grad, grad_temperature=m.temperature.grad)
        return total

    def step_single(q, v, mask, record=False):
        return api_step(model, q, v, mask, record)

    class TimedKernels(CudaKernels):
        """The product kernels, with CUDA events around the forward call (for the roofline entry)."""
        record = False

        def maxmean_fwd(self, q, v, scale, T_):
            if not self.record:
                return super().maxmean_fwd(q, v, scale, T_)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = super().maxmean_fwd(q, v, scale, T_)
            e1.record(); fwd_ev.append((e0, e1))
            return out

    timed_kernels = TimedKernels()

    def step_sharded(q, v, mask, record=False):
        timed_kernels.record = record
        out = sharded_contrastive_step(q, v, T, mask, kernels=timed_kernels)
        return out["loss"]

    step = step_single if world == 1 else step_sharded
    for s in sets:
        s[0].requires_grad_(world == 1); s[1].requires_grad_(world == 1)

    # ---- device-resident arm -------------------------------------------------------------------
    for i in range(args.warmup):
        step(*sets[i % n_sets])
    launches0 = lib.triad_launch_count()
    with ClockSampler(local) as clocks:
        ms = timed(lambda i: step(*sets[i % n_sets], record=True), args.steps)
    gpu_launches = int(lib.triad_launch_count() - launches0)     # libtriad_b200.so kernels inside the timed region (this rank)
    value = float(B) * B / (ms * 1e-3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_step)

    # ---- end-to-end arm: pinned host inputs -> H2D -> step -> loss D2H --------------------------
    # Every step's embeddings start in PINNED HOST memory and its loss is read back on the host.  As in any
    # input pipeline, the H2D copy of step i+1 is issued on a copy stream while step i computes (double
    # buffered device staging); each step still pays for its own copy and its own D2H read inside the timed
    # region, but copy and compute overlap instead of serialising.
    host = [(q.detach().cpu().pin_memory(), v.detach().cpu().pin_memory(),
             None if m is None else m.cpu().pin_memory()) for (q, v, m) in sets]
    d2h = {"bytes": 0}
    copy_stream = torch.cuda.Stream(device=dev)
    staged = {}

    def issue_copy(i):
        hq, hv, hm = host[i % n_sets]
        with torch.cuda.stream(copy_stream):
            q = hq.to(dev, non_blocking=True)
            v = hv.to(dev, non_blocking=True)
            m = None if hm is None else hm.to(dev, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        staged[i] = (q, v, m, ev)

    # The loss of every step is copied to PINNED host memory (D2H, 4 bytes) on the compute stream and read on the
    # host one step later — after the next step has been queued — so the device never idles waiting for Python,
    # exactly like a training loop that logs the loss with a one-step lag.  Every step's value is read inside the
    # timed region (the last one before the closing synchronise).
    loss_host = [torch.zeros((), dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_ev = [torch.cuda.Event(), torch.cuda.Event()]
    seen = {"n": 0, "last": None}

    def e2e_step(i):
        if i not in staged:
            issue_copy(i)
        q, v, m, ev = staged.pop(i)
        torch.cuda.current_stream().wait_event(ev)
        for t in (q, v, m):
            if t is not None:
                t.record_stream(torch.cuda.current_stream())
        issue_copy(i + 1)                     # next step's inputs travel while this step computes
        q.requires_grad_(world == 1); v.requires_grad_(world == 1)
        loss = step(q, v, m)
        loss_host[i % 2].copy_(loss.detach().float(), non_blocking=True)      # D2H read of the step's result
        loss_ev[i % 2].record()
        d2h["bytes"] = 4
        if i > 0:                             # consume the previous step's loss on the host
            loss_ev[(i - 1) % 2].synchronize()
            seen["last"] = float(loss_host[(i - 1) % 2]); seen["n"] += 1

    def e2e_run(K):
        staged.clear()
        seen["n"] = 0
        for i in range(K):
            e2e_step(i)
        loss_ev[(K - 1) % 2].synchronize()
        seen["last"] = float(loss_host[(K - 1) % 2]); seen["n"] += 1
        assert seen["n"] == K and seen["last"] == seen["last"]      # K losses read on the host, finite
        staged.clear()                        # the look-ahead copy issued by the last step is not used

    if args.warmup > 0:
        e2e_run(min(args.warmup, 3))
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    e2e_run(args.steps)
    e1.record()
    sync_all()
    e2e_t = torch.tensor([e0.elapsed_time(e1) / args.steps], device=dev)
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_ms = e2e_t.item()
    h2d = in_bytes + (host[0][2].numel() * 8 if host[0][2] is not None else 0)
    del host, staged
    tokens_local = int(sets[0][2].sum().item()) if cfg["masked"] else Bl * cfg["Nq"]

    # ---- roofline of the dominant kernel (tcgen05 forward) and of the step ------------------------------------
    def roofline_block(fwd_ms, step_ms, Bcols, tokens, Nv, D, nranks=1, traffic=None):
        f_fwd, f_bwd = algorithmic_flops(Bcols, tokens, Nv, D)
        achieved = f_fwd / (fwd_ms * 1e-3) / 1e12
        return {"bound": "tensor", "kernel": "maxmean_tc_kernel (fwd call: memset + kernel + finalize_clip)",
                "achieved": achieved, "peak": peaks["bf16"], "unit": "TFLOP/s", "frac": achieved / peaks["bf16"],
                "peak_source": f"{peaks['source']}: burst; sustained {peaks['bf16_sustained']}",
                "frac_of_sustained": achieved / peaks["bf16_sustained"], "ms": fwd_ms, "traffic": traffic,
                "algorithmic_flops_per_launch": f_fwd, "step_flops": f_fwd + f_bwd,
                "step_frac_of_peak": (f_fwd + f_bwd) / (step_ms * 1e-3) / 1e12 / peaks["bf16"],
                "step_frac_of_sustained_peak": (f_fwd + f_bwd) / (step_ms * 1e-3) / 1e12 / peaks["bf16_sustained"]}

    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        traffic = json.load(open(tpath)).get(cfg_key)
    roof = None
    if fwd_ev:
        fwd_ms = statistics.mean(a.elapsed_time(b) for a, b in fwd_ev)
        roof = roofline_block(fwd_ms, ms, B, tokens_local, cfg["Nv"], cfg["D"], world, traffic)
    fwd_ev.clear()

    extras = {}
    if world == 1 and not args.no_extras and cfg_key == "cfg2":
        # ---- burst vs. sustained: the same step, 60 back to back from an idle GPU, timed one by one (DESIGN.md §4) ----
        torch.cuda.synchronize()
        time.sleep(2.0)
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(61)]
        with ClockSampler(local) as ck:
            evs[0].record()
            for i in range(60):
                step(*sets[i % n_sets])
                evs[i + 1].record()
            torch.cuda.synchronize()
        per = [evs[i].elapsed_time(evs[i + 1]) for i in range(60)]
        f_all = sum(algorithmic_flops(B, tokens_local, cfg["Nv"], cfg["D"]))
        extras["burst_vs_sustained"] = {
            "what": "60 steps back to back after 2 s of idle, each step timed with its own CUDA events: the first ~50 ms run at "
                    "boost clocks, then the power governor (sw_power_cap) lowers the SM clock for the whole step",
            "first_10_steps_ms": sum(per[1:11]) / 10, "last_10_steps_ms": sum(per[-10:]) / 10,
            "first_10_frac_of_burst_peak": f_all / (sum(per[1:11]) / 10 * 1e-3) / 1e12 / peaks["bf16"],
            "last_10_frac_of_sustained_peak": f_all / (sum(per[-10:]) / 10 * 1e-3) / 1e12 / peaks["bf16_sustained"],
            "per_step_ms": [round(x, 3) for x in per], "clocks": ck.summary()}
    if world == 1 and not args.no_extras:
        # ---- the reference's FULL loss (contrastive + regularisers, SURVEY §8 f1), reported beside the metric ----
        model.triad_regularizers = True
        for i in range(2):
            step(*sets[i % n_sets])
        torch.cuda.synchronize()
        time.sleep(1.0)                       # every side block starts from an idle GPU, as the headline region does
        k_full = max(3, min(args.steps, 10))
        # timed like every other block (one pair of events around K steps); in addition every step gets its own event
        # and the host notes when it had finished queueing it, so a slow step can be told from a late host
        ev_full = [torch.cuda.Event(enable_timing=True) for _ in range(k_full + 1)]
        host_t = []

        def full_step(i):
            if i == 0:
                ev_full[0].record()
            t0 = time.perf_counter()
            step(*sets[i % n_sets])
            host_t.append((time.perf_counter() - t0) * 1e3)
            ev_full[i + 1].record()

        with ClockSampler(local) as ck:
            full_ms = timed(full_step, k_full)
        per_full = [ev_full[i].elapsed_time(ev_full[i + 1]) for i in range(k_full)]
        model.triad_regularizers = False
        extras["full_loss"] = {
            "value": float(B) * B / (full_ms * 1e-3), "unit": "clip-pairs/s", "ms_per_step": full_ms, "steps": k_full,
            "per_step_ms": [round(x, 2) for x in per_full], "median_ms": statistics.median(per_full),
            "host_queue_ms_per_step": [round(x, 2) for x in host_t],
            "clocks": ck.summary(),
            "what": "same step with the reference's regularisers on (model.py:394-428 / :516-542): dense non-negative "
                    "pressure, smoothness / sparsity on the positive pairs; not part of BASELINE.json's metric"}
        del sets
        torch.cuda.empty_cache()

        # ---- cfg 3: ragged text queries (masked mean), B=512 ----------------------------------------------------
        if cfg_key != "cfg3":
            c3 = CONFIGS["cfg3"]
            s3 = make_device_inputs(c3, c3["B"], 777, dev, 3)
            for s in s3:
                s[0].requires_grad_(True); s[1].requires_grad_(True)
            for i in range(3):
                step_single(*s3[i % 3])
            torch.cuda.synchronize()
            time.sleep(1.0)
            fwd_ev.clear()
            k3 = max(5, min(args.steps, 20))
            with ClockSampler(local) as ck:
                ms3 = timed(lambda i: step_single(*s3[i % 3], record=True), k3)
            tok3 = float(sum(int(s[2].sum().item()) for s in s3)) / 3.0
            fwd3 = statistics.mean(a.elapsed_time(b) for a, b in fwd_ev)
            fwd_ev.clear()
            extras["cfg3"] = {"workload": c3["name"], "ms_per_step": ms3, "steps": k3,
                              "value": float(c3["B"]) ** 2 / (ms3 * 1e-3), "unit": "clip-pairs/s", "clocks": ck.summary(),
                              "valid_tokens_per_step": tok3,
                              "roofline": roofline_block(fwd3, ms3, c3["B"], tok3, c3["Nv"], c3["D"], 1,
                                                         json.load(open(tpath)).get("cfg3") if os.path.exists(tpath) else None),
                              "note": "flops count VALID tokens only (padded tokens are packed out before the tensor cores)"}
            del s3
            torch.cuda.empty_cache()

        # ---- cfg 4: one rank's share (1024 x 8192), then the whole B=8192 step, on ONE GPU ------------------------
        c4 = CONFIGS["cfg4"]
        Bq4, Bv4 = c4["B"] // 8, c4["B"]
        (q4, _, _), = make_device_inputs(c4, Bv4, 99, dev, 1)
        (_, v4, _), = make_device_inputs(c4, Bv4, 98, dev, 1)
        T4 = torch.tensor(1.5, device=dev)
        ck4 = CudaKernels()
        q4r = q4[:Bq4].contiguous()

        def rank_step():
            sc = ck4.row_scale(None, Bq4, c4["Nq"], dev)
            clip4, idx4 = ck4.maxmean_fwd(q4r, v4, sc, T4)
            lse4, cp4 = ck4.infonce_partial(clip4, Bv4, 0)
            g4, _ = ck4.infonce_finish(clip4, Bv4, 0, lse4, cp4.reshape(1, 2, Bv4))
            return ck4.maxmean_bwd(q4r, v4, idx4, g4, clip4, sc, T4)

        rank_step()
        with ClockSampler(local) as ck:
            rs_ms = timed(lambda i: rank_step(), 2)
        extras["cfg4_rank_shape_1gpu"] = {
            "workload": f"one rank's share of cfg4 at 8 GPUs: {Bq4} queries x {Bv4} images, fwd + InfoNCE block + bwd, no collectives",
            "ms_per_step": rs_ms, "value": float(Bq4) * Bv4 / (rs_ms * 1e-3), "unit": "clip-pairs/s per GPU", "clocks": ck.summary()}
        del q4r
        if not args.no_cfg4_1gpu:
            m4 = triad_b200.TriadHotPath(temperature=1.5).to(dev)
            m4.triad_regularizers = False
            q4.requires_grad_(True); v4.requires_grad_(True)
            api_step(m4, q4, v4, None)                       # warm-up (allocates the 17 GB argmax buffer once)
            fwd_ev.clear()
            with ClockSampler(local) as ck:
                ms4 = timed(lambda i: api_step(m4, q4, v4, None, record=True), 2)
            fwd4 = statistics.mean(a.elapsed_time(b) for a, b in fwd_ev)
            fwd_ev.clear()
            extras["cfg4_1gpu"] = {
                "workload": "cfg4 on ONE GPU: B=8192 x 8192, 250 x 256, D=512, bf16, fwd + InfoNCE + bwd through the drop-in API "
                            "(the strong-scaling denominator of the N>1 lines)",
                "ms_per_step": ms4, "steps": 2, "value": float(c4["B"]) ** 2 / (ms4 * 1e-3), "unit": "clip-pairs/s",
                "clocks": ck.summary(),
                "roofline": roofline_block(fwd4, ms4, c4["B"], c4["B"] * c4["Nq"], c4["Nv"], c4["D"])}
            q4.grad = v4.grad = None
            del m4
        del q4, v4
        torch.cuda.empty_cache()

        # ---- f3: the fused projection head on the audio shape of cfg 2 (64 000 HuBERT frames, 768 -> 512 -> 512) -----
        extras["f3_projection_head"] = f3_block(dev, local, peaks, timed)

        # ---- cfg 5: one query against a 104.9 GB gallery, forward-only top-k (HBM-bound for text queries) ---------
        if not args.no_cfg5:
            extras["cfg5"] = cfg5_block(dev, local, peaks, 1, 0, timed)

    if world > 1 and not args.no_extras and not args.no_cfg5:
        extras["cfg5_sharded"] = cfg5_block(dev, local, peaks, world, rank, timed)

    out = None
    if rank == 0:
        out = {
            "metric": "clip-pairs/sec", "value": value, "unit": "clip-pairs/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": cfg["name"], "global_batch": B, "rows_per_rank": Bl,
                       "parallelism": f"row-sharded x{world}" if world > 1 else "single GPU",
                       "l2": f"{n_sets} rotating input sets ({n_sets * in_bytes / 2**20:.0f} MiB) > 126 MB L2, "
                             "so every step reads its embeddings from HBM",
                       "scaling_note": "N=1 runs cfg 2 (the configuration the metric is quoted on); N>1 runs cfg 4 with the TOTAL "
                                       "work fixed (B=8192), i.e. strong scaling among the N>1 lines; the same B=8192 step on one "
                                       "GPU is the `cfg4_1gpu` block of the N=1 line"},
            "clocks": clocks.summary(),
            "e2e": {"value": float(B) * B / (e2e_ms * 1e-3), "unit": "clip-pairs/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h["bytes"],
                    "pipeline": "pinned-host inputs of step i+1 are copied (copy stream) while step i computes; each "
                                "step's loss is copied to pinned host memory and read on the host one step later"},
            "gpu_launches": gpu_launches,
            "roofline": roof,
        }
        if parity is not None:
            out.update({"parity_nranks": parity["parity_nranks"], "parity": parity["parity"], "parity_detail": parity})
        out.update(extras)
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline(cfg, args.cpu_seconds)
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return out


def f3_block(dev, local, peaks, timed):
    """SURVEY §8 f3: projection2(layer_norm(projection1(x))) for B=256 x 250 frames, Din=768, as one launch
    (triad_project_tokens), next to torch.nn's three kernels under autocast on the same weights."""
    import torch
    from triad_b200.producers import ProjectionHead
    B, N, Din, Dout = 256, 250, 768, 512
    torch.manual_seed(3)
    head = ProjectionHead(Din, Dout).to(dev)
    xs = [torch.randn(B, N, Din, device=dev).bfloat16() for _ in range(3)]

    def torch_head(x):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            return head.projection2(head.layer_norm(head.projection1(x)))

    with torch.no_grad():
        y = head(xs[0]); ref = torch_head(xs[0])
        err = ((y.float() - ref.float()).norm() / ref.float().norm()).item()
        for i in range(3):
            head(xs[i])
        with ClockSampler(local) as ck:
            ms = timed(lambda i: head(xs[i % 3]), 30)
        for i in range(3):
            torch_head(xs[i])
        ms_t = timed(lambda i: torch_head(xs[i % 3]), 30)
    flops = 2.0 * B * N * (Din * 512 + 512 * Dout)
    return {"workload": f"projection head, {B}x{N} tokens, {Din} -> 512 -> LayerNorm -> {Dout}, bf16, one launch",
            "ms": ms, "tflops": flops / (ms * 1e-3) / 1e12, "frac_of_bf16_peak": flops / (ms * 1e-3) / 1e12 / peaks["bf16"],
            "torch_nn_autocast_ms": ms_t, "rel_err_vs_torch_nn_autocast": err, "clocks": ck.summary()}


def cfg5_block(dev, local, peaks, world, rank, timed):
    """cfg 5: one query (77 text tokens / 250 audio frames) against 100 000 images x 1024 patches (104.9 GB bf16).
    world == 1: the whole gallery on this GPU.  world > 1: the gallery sharded by images over the ranks, local top-k,
    all-gather of k (score, id) pairs, merge (triad_b200.dist.sharded_retrieve_topk)."""
    import torch
    from triad_b200 import retrieval as R
    n_img, Nv, D, k = CFG5["n_img"], CFG5["Nv"], CFG5["D"], CFG5["k"]
    n_loc = n_img // world + (1 if rank < n_img % world else 0)
    id0 = rank * (n_img // world) + min(rank, n_img % world)
    gal = torch.empty(n_loc, Nv, D, dtype=torch.bfloat16, device=dev)
    g = torch.Generator(device=dev).manual_seed(7 + rank)
    step_imgs = max(1, (1 << 30) // (Nv * D * 2))                       # fill 1 GiB at a time
    for i in range(0, n_loc, step_imgs):
        blk = torch.randn(min(step_imgs, n_loc - i), Nv, D, generator=g, device=dev, dtype=torch.float32)
        gal[i:i + blk.shape[0]] = torch.nn.functional.normalize(blk, dim=2).to(torch.bfloat16)
        del blk
    gq = torch.Generator(device=dev).manual_seed(11)                    # the same query on every rank
    res = {"workload": CFG5["name"] + (f", gallery sharded over {world} ranks" if world > 1 else ""),
           "gallery_bytes": float(n_img) * Nv * D * 2, "queries": {}}
    for name, Nq in (("text77", 77), ("audio250", 250)):
        q = torch.nn.functional.normalize(torch.randn(Nq, D, generator=gq, device=dev), dim=1).to(torch.bfloat16)
        if world > 1:
            from triad_b200.dist import sharded_retrieve_topk
            fn = lambda i: sharded_retrieve_topk(q, gal, 1.5, k, id0)           # noqa: E731
        else:
            fn = lambda i: R.retrieve_topk(q, gal, 1.5, k)                       # noqa: E731
        s, ids = fn(0)
        with ClockSampler(local) as ck:
            ms = timed(fn, 5)
        # spot check of the winner against a plain fp32 evaluation (on the rank that owns it)
        j = int(ids[0]) - id0
        chk = None
        if 0 <= j < n_loc:
            ref = ((q.float() @ gal[j].float().t()) / 1.5).max(dim=1).values.mean().item()
            chk = abs(ref - s[0].item())
        gbs = res["gallery_bytes"] / (ms * 1e-3) / 1e9
        flops = 2.0 * Nq * n_img * Nv * D
        bound = "hbm" if Nq < peaks["bf16"] * 1e3 / peaks["hbm"] else "tensor/hbm (balanced)"
        res["queries"][name] = {
            "Nq": Nq, "ms_per_query": ms, "queries_per_s": 1e3 / ms, "clocks": ck.summary(), "top1_fp32_check_abs_err": chk,
            "roofline": {"bound": bound, "achieved": gbs, "peak": peaks["hbm"] * world, "unit": "GB/s",
                         "frac": gbs / (peaks["hbm"] * world), "algorithmic_bytes_per_launch": res["gallery_bytes"],
                         "tflops": flops / (ms * 1e-3) / 1e12, "peak_source": peaks["source"]}}
    del gal
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="triad", choices=["triad", "reference"])
    ap.add_argument("--config", default="auto", choices=["auto"] + list(CONFIGS))
    ap.add_argument("--verify", action="store_true", help="only the N-rank parity check (sharded vs single-GPU vs oracle)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the cfg3 / cfg4 / cfg5 / full-loss blocks")
    ap.add_argument("--no-cfg4-1gpu", action="store_true", help="skip the B=8192 single-GPU step (about 20 s)")
    ap.add_argument("--no-cfg5", action="store_true", help="skip the 104.9 GB retrieval block")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned as DIR/<name>.npy (single GPU, --impl triad)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus != world and world > 1:
        args.gpus = world
    if args.dump_outputs and (max(args.gpus, world) > 1 or args.impl != "triad" or args.verify):
        ap.error("--dump-outputs needs --gpus 1 and --impl triad, without --verify")
    cfg_key = args.config if args.config != "auto" else ("cfg2" if max(args.gpus, world) == 1 else "cfg4")
    if args.impl == "reference":
        run_reference(args, cfg_key)
    else:
        if args.gpus > 1 and world == 1:
            raise SystemExit("for --gpus N > 1 launch with: python -m torch.distributed.run --nnodes=1 "
                             "--nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...")
        run_triad(args, cfg_key)


if __name__ == "__main__":
    main()
