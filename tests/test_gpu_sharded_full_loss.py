"""GPU tier: the row-sharded full-loss step and the two library additions it is built on —
triad_dense_grad_gemm_f32 (fp32 output, optionally added to) and TRIAD_BWD_ACCUMULATE_DV — against fp32 matmuls,
the plain backward and the single-GPU drop-in full loss; with >= 2 GPUs, the torchrun check of
tools/sharded_full_loss_check.py."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

GEMM_SHAPES = [
    # M (rows of N), Kc (columns of N), D
    (300, 1536, 512),          # row / K tails
    (1000, 520, 256),          # one N half, Kc % 64 != 0
    (77, 200, 64),             # tiny: partial tiles everywhere
    (256, 4096, 512),          # mode 0: one row tile, many K splits
    (2500, 264, 128),          # mode 1: two row tiles, many K splits
]


def _rel(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return ((a - b).norm() / b.norm()).item()


@pytest.mark.parametrize("shape", GEMM_SHAPES, ids=["x".join(map(str, s)) for s in GEMM_SHAPES])
@pytest.mark.parametrize("mode", [0, 1])
def test_dense_grad_gemm_f32_modes(shape, mode):
    from triad_b200 import ops
    M, Kc, D = shape
    g = torch.Generator().manual_seed(M + Kc + D + mode)
    N = (torch.randn(M, Kc, generator=g) * 0.05).bfloat16().cuda()
    x = torch.randn(Kc if mode == 0 else M, D, generator=g).bfloat16().cuda()
    ref = (N.float() @ x.float()) if mode == 0 else (N.float().t() @ x.float())
    out = torch.full_like(ref, float("nan"))
    ops.dense_grad_gemm_f32(N, x, mode, out, False)
    assert _rel(out, ref) < 1e-5
    # bf16 of the fp32 result is the bf16 entry point's output, bit for bit
    assert torch.equal(out.bfloat16(), ops.dense_grad_gemm(N, x, mode))
    # accumulate onto zeros == plain; onto a random prior == prior + product (one fp32 add)
    acc = torch.zeros_like(ref)
    ops.dense_grad_gemm_f32(N, x, mode, acc, True)
    assert torch.equal(acc, out)
    prior = torch.randn(ref.shape, generator=g).cuda()
    acc = prior.clone()
    ops.dense_grad_gemm_f32(N, x, mode, acc, True)
    assert torch.equal(acc, prior + out)
    assert _rel(acc, prior.double() + ref.double()) < 1e-5


def test_dense_grad_gemm_f32_into_rows_of_a_larger_buffer():
    """dV of one image chunk written straight into its rows of a [Bv*Nv, D] buffer, N read through a row pitch larger
    than the chunk's width; the rows around it stay untouched."""
    from triad_b200 import ops
    M, Kc, D, r0 = 500, 768, 512, 1024
    g = torch.Generator().manual_seed(3)
    big_n = (torch.randn(M, Kc + 256, generator=g) * 0.05).bfloat16().cuda()
    N = big_n[:, :Kc]
    q2 = torch.randn(M, D, generator=g).bfloat16().cuda()
    buf = torch.randn(4096, D, generator=g).cuda()
    before = buf.clone()
    ops.dense_grad_gemm_f32(N, q2, 1, buf[r0:r0 + Kc], False)
    assert torch.equal(buf[:r0], before[:r0]) and torch.equal(buf[r0 + Kc:], before[r0 + Kc:])
    assert _rel(buf[r0:r0 + Kc], N.float().t() @ q2.float()) < 1e-5


@pytest.mark.parametrize("case", ["bf16", "bf16_generic_dv", "bf16_small_blocks", "fp32"])
def test_bwd_accumulate_dv(case):
    from triad_b200 import _lib, ops
    dt = torch.float32 if case == "fp32" else torch.bfloat16
    Bq, Bv, Nq, Nv, D = 24, 20, 50, 64, 256
    g = torch.Generator().manual_seed(7)
    q = (torch.randn(Bq, Nq, D, generator=g) / D ** 0.5).to(dt).cuda()
    v = (torch.randn(Bv, Nv, D, generator=g) / D ** 0.5).to(dt).cuda()
    T = torch.tensor(1.5, device="cuda")
    scale = ops.row_scale(None, Bq, Nq, q.device)
    _, idx = ops.maxmean_fwd(q, v, scale, T)
    gr = (torch.randn(Bq, Bv, generator=g) * 0.01).cuda()
    flags = {"bf16": 0, "bf16_generic_dv": _lib.BWD_GENERIC_DV, "bf16_small_blocks": _lib.BWD_SMALL_BLOCKS, "fp32": 0}[case]
    _, dv0, _ = ops.maxmean_bwd(q, v, idx, gr, None, scale, T, need_dq=False, need_dT=False, dv_f32=True, flags=flags)
    zero = torch.zeros(Bv, Nv, D, device="cuda")
    ops.maxmean_bwd(q, v, idx, gr, None, scale, T, need_dq=False, need_dT=False, flags=flags | _lib.BWD_ACCUMULATE_DV,
                    dv_out=zero)
    assert torch.equal(zero, dv0)
    prior = torch.randn(Bv, Nv, D, generator=g).cuda() * dv0.abs().max()
    acc = prior.clone()
    ops.maxmean_bwd(q, v, idx, gr, None, scale, T, need_dq=False, need_dT=False, flags=flags | _lib.BWD_ACCUMULATE_DV,
                    dv_out=acc)
    # Each query block's contribution is added with one fp32 rounding relative to the running sum, in both calls.  The
    # same backward on |q|, |g| is the sum of the contributions' magnitudes, which bounds every partial sum; the query
    # blocks number at most Bq (64 KB blocks of 50 x 256 bf16 rows: 2 queries each, 12 blocks, with SMALL_BLOCKS).
    _, dv_abs, _ = ops.maxmean_bwd(q.abs(), v, idx, gr.abs(), None, scale, T, need_dq=False, need_dT=False, dv_f32=True,
                                   flags=flags)
    n_blocks = Bq if case == "bf16_small_blocks" else 1
    want = prior.double() + dv0.double()
    tol = (n_blocks + 2) * torch.finfo(torch.float32).eps * (prior.abs().double() + 1.01 * dv_abs.double()) + 1e-30
    assert bool(((acc.double() - want).abs() <= tol).all())
    if dt == torch.bfloat16:                  # a bf16 dv has nothing to accumulate into in fp32: refused
        with pytest.raises(_lib.TriadError):
            ops.maxmean_bwd(q, v, idx, gr, None, scale, T, need_dq=False, need_dT=False, flags=_lib.BWD_ACCUMULATE_DV)


class _Recording:
    """CudaKernels that keeps the argmax buffer the step hands to the dq backward."""

    def __new__(cls):
        from triad_b200.dist import CudaKernels

        class K(CudaKernels):
            def maxmean_bwd_dq(self, q, v, idx, g, scale, T):
                self.idx = idx
                return super().maxmean_bwd_dq(q, v, idx, g, scale, T)
        return K()


def _inputs(kind, B, Nq, Nv, D, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    q = (torch.randn(B, Nq, D, generator=g, device="cuda") * 2 / D ** 0.5).bfloat16()
    v = (torch.randn(B, Nv, D, generator=g, device="cuda") * 2 / D ** 0.5).bfloat16()
    mask = None
    if kind == "tv":
        lens = torch.randint(8, Nq + 1, (B,), generator=g, device="cuda")
        lens[0] = Nq
        mask = (torch.arange(Nq, device="cuda")[None, :] < lens[:, None]).to(torch.int64)
    return q, v, mask


def _dropin(kind, q, v, mask, T, thr, w):
    import triad_b200
    m = triad_b200.TriadHotPath(T, thr, w).cuda()
    qd, vd = q.clone().requires_grad_(), v.clone().requires_grad_()
    if kind == "av":
        clip, tok = m.compute_all_similarities_av(qd, vd)
        assert tok.nonneg is not None                              # the merged forward
        total, con, reg, smooth, stats = m.compute_contrastive_loss_av(clip, tok)
    else:
        clip, tok = m.compute_all_similarities_tv(qd, vd, mask)
        assert tok.nonneg is not None
        total, stats = m.compute_contrastive_loss_tv(clip, tok)
        con = reg = smooth = None
    idx, clip32 = tok.idx_t.clone(), tok.clip.detach().clone()
    total.backward()
    return {"total": total.item(), "contrastive": None if con is None else con.item(),
            "reg": None if reg is None else reg.item(), "smooth": None if smooth is None else smooth.item(),
            "stats": dict(stats), "clip": clip32, "idx": idx, "dq": qd.grad.float(), "dv": vd.grad.float(),
            "dT": m.temperature.grad.item()}


@pytest.mark.parametrize("chunks", ["one", "several"])
@pytest.mark.parametrize("kind", ["av", "tv"])
def test_single_rank_matches_dropin_full_loss(kind, chunks):
    from triad_b200.dist import sharded_full_loss_step, stats_from_all_sums
    B, Nq, Nv, D = (48, 250, 256, 512) if kind == "av" else (64, 77, 256, 512)
    T, thr, w = 0.8, 0.01, 0.5                       # T < 1: the calibration term is active
    q, v, mask = _inputs(kind, B, Nq, Nv, D, 11)
    ref = _dropin(kind, q, v, mask, T, thr, w)
    per_image = B * Nq * Nv * 2
    chunk_bytes = None if chunks == "one" else 17 * per_image      # 17 + 17 + the rest: a short last chunk
    k = _Recording()
    out = sharded_full_loss_step(q, v, torch.tensor(T, device="cuda"), kind, mask, kernels=k,
                                 patch_sparsity_threshold=thr, patch_sparsity_weight=w, chunk_bytes=chunk_bytes)
    torch.cuda.synchronize()
    assert torch.equal(out["clip_rows"], ref["clip"])
    assert torch.equal(k.idx, ref["idx"])
    assert abs(out["total"].item() - ref["total"]) <= 1e-5 * abs(ref["total"])
    if kind == "av":
        for key in ("contrastive", "reg", "smooth"):
            assert abs(out[key].item() - ref[key]) <= 1e-5 * abs(ref[key]), key
    else:
        assert abs((out["contrastive"] + out["reg"]).item() - ref["total"]) <= 1e-5 * abs(ref["total"])
    stats = stats_from_all_sums(out["all_sums"], B, kind)
    for key, val in ref["stats"].items():
        assert abs(stats[key] - val) <= 1e-6 * max(1.0, abs(val)), key
    assert _rel(out["dq"], ref["dq"]) < 4e-3
    assert _rel(out["dv"], ref["dv"]) < 4e-3
    assert abs(out["dT"].item() - ref["dT"]) <= 1e-4 * abs(ref["dT"])
    assert abs(out["dT_global"].item() - ref["dT"]) <= 1e-4 * abs(ref["dT"])


@pytest.mark.parametrize("case", ["patch_dropout_bf16", "fp32"])
def test_fallback_shapes_match_the_composed_pair(case):
    """Shapes the merged pass does not take run the two separate calls behind the same interface."""
    from triad_b200.dist import sharded_contrastive_step, sharded_full_loss_step, sharded_regularizer_step
    if case == "patch_dropout_bf16":
        q, v, _ = _inputs("av", 16, 50, 203, 512, 5)
    else:
        q, v, _ = _inputs("av", 8, 20, 40, 64, 6)
        q, v = q.float(), v.float()
    T = torch.tensor(0.8, device="cuda")
    out = sharded_full_loss_step(q, v, T, "av")
    con = sharded_contrastive_step(q, v, T)
    reg = sharded_regularizer_step(q, v, T, "av")
    assert torch.equal(out["total"], con["loss"] + reg["reg"])
    assert torch.equal(out["smooth"], reg["smooth"])
    assert torch.equal(out["dq"], (con["dq"].float() + reg["dq"].float()).to(q.dtype))
    assert torch.equal(out["dv"], (con["dv"].float() + reg["dv"].float()).to(v.dtype))
    assert torch.equal(out["dT"], con["dT"] + reg["dT"])


def test_autograd_face_on_cuda():
    """sharded_full_loss: backward of 2.5*total scales the eager gradients by 2.5 on the device."""
    from triad_b200 import regularizers as R
    from triad_b200.dist import sharded_full_loss, sharded_full_loss_step
    q, v, _ = _inputs("av", 16, 50, 256, 512, 8)
    T = torch.tensor(0.8, device="cuda")
    eager = sharded_full_loss_step(q, v, T, "av")
    qd, vd, Td = q.clone().requires_grad_(), v.clone().requires_grad_(), T.clone().requires_grad_()
    total, con, reg, smooth, stats = sharded_full_loss(qd, vd, Td, "av")
    assert torch.equal(total, eager["total"]) and not con.requires_grad
    (2.5 * total).backward()
    two5 = torch.tensor(2.5, device="cuda")
    assert torch.equal(qd.grad, R.scale_by(eager["dq"], two5))
    assert torch.equal(vd.grad, R.scale_by(eager["dv"], two5))
    assert torch.equal(Td.grad, eager["dT"] * 2.5)
    assert "av_hardest_negative" in stats


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least 2 GPUs")
def test_sharded_full_loss_under_nccl():
    n = 2 if torch.cuda.device_count() < 8 else 8
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
           "--master-addr", "127.0.0.1", "--master-port", "29519", os.path.join("tools", "sharded_full_loss_check.py")]
    r = subprocess.run(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "SHARDED_FULL_LOSS_OK" in r.stdout
