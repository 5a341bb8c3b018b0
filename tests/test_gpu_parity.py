"""GPU tier: the CUDA path, called through the drop-in methods (-> ctypes -> C ABI), against
(1) the golden vectors of the unmodified reference and (2) the CPU oracle, plus size-independent
properties at the full BASELINE cfg-2 shape.

Tolerances are the north star's: argmax indices bit-exact; loss / similarity / gradients within
1e-4 relative for fp32 inputs and 1e-2 for bf16 inputs.
"""
import math

import numpy as np
import pytest
import torch

from oracle import oracle as O
from oracle.cases import CASES, build_inputs, projection
from tests.helpers import certify_near_ties, check_inputs_reproduce, load_golden, rel_err

pytestmark = pytest.mark.gpu

FWD_SIMT, FWD_1CTA, FWD_SYNC = 1, 2, 8


def _model(T, flags=0, regularizers=False):
    """regularizers=False: the fused contrastive path on its own (what most tests pin); True: the full loss."""
    import triad_b200
    # the two patch_sparsity_* values are the ones oracle/gen_golden.py gave the reference's methods
    m = triad_b200.TriadHotPath(temperature=T, patch_sparsity_threshold=0.80, patch_sparsity_weight=0.01).cuda()
    m.triad_fwd_flags = flags
    m.triad_regularizers = regularizers
    return m


def _run_case(case, flags):
    q, v, mask, T = build_inputs(case)
    m = _model(T, flags)
    qd, vd = q.cuda().requires_grad_(), v.cuda().requires_grad_()
    if case.kind == "av":
        clip, tok = m.compute_all_similarities_av(qd, vd)
        total, con, reg, smooth, stats = m.compute_contrastive_loss_av(clip, tok)
    else:
        clip, tok = m.compute_all_similarities_tv(qd, vd, mask.cuda())
        con, stats = m.compute_contrastive_loss_tv(clip, tok)
    con.backward()
    torch.cuda.synchronize()
    return q, v, mask, T, m, qd, vd, clip, tok, con, stats


def _variants(case):
    if case.dtype == "fp32":
        return [0]
    return [0, FWD_1CTA, FWD_SIMT]        # tcgen05 cta_group::2, cta_group::1, CUDA-core


ALL = [(c, f) for c in CASES for f in _variants(c)]


@pytest.mark.parametrize("case,flags", ALL, ids=[f"{c.name}-f{f}" for c, f in ALL])
def test_golden_parity(case, flags):
    gold = load_golden(case.name)
    q, v, mask, T, m, qd, vd, clip, tok, con, stats = _run_case(case, flags)
    check_inputs_reproduce(gold, q, v)
    fp32 = case.dtype == "fp32"
    tol = 1e-4 if fp32 else 1e-2

    # (1) argmax patch indices: bit-exact against the reference's torch.max
    assert tok.shape == (case.B, case.B, case.Nq, case.Nv)
    assert np.array_equal(tok.argmax().cpu().numpy(), gold["idx"].astype(np.int64))

    # (2) clip similarity: same dtype as the reference returns, values within tolerance
    assert clip.dtype == (torch.bfloat16 if bool(gold["clip_is_bf16"]) else torch.float32)
    assert rel_err(clip.float().cpu(), gold["clip"]) < tol
    oracle = O.contrastive_step_closed_form(q, v, T, mask)
    # fp32 clip vs the oracle's fp32 clip.  bf16: the tensor core and the CPU accumulate the 512-term dot
    # products in different orders, so an accumulator that sits on a bf16 rounding boundary can round the
    # other way: that moves ONE row maximum by one bf16 ulp (2^-8 relative), i.e. one clip element by
    # ~2^-8/Nq.  A handful of such flips gives ~1e-5 norm-wise; the north star's bound is 1e-2.
    ctol = 2e-6 if fp32 else 5e-5
    assert rel_err(tok.clip.detach().cpu(), oracle["clip"]) < ctol

    # (3) loss and gradients vs the reference
    assert abs(con.item() - float(gold["contrastive"])) <= tol * abs(float(gold["contrastive"]))
    P = projection(case)
    dq = qd.grad.double().cpu() @ P if P is not None else qd.grad.double().cpu()
    dv = vd.grad.double().cpu() @ P if P is not None else vd.grad.double().cpu()
    assert qd.grad.dtype == q.dtype and vd.grad.dtype == v.dtype
    assert rel_err(dq, gold["dq"]) < tol
    assert rel_err(dv, gold["dv"]) < tol
    scale = (oracle["g"].abs() * oracle["clip"].abs().double()).sum().item() / T
    assert abs(m.temperature.grad.item() - float(gold["dT"])) < (1e-4 if fp32 else 2e-2) * scale

    # (4) and vs the fp64 oracle (tighter: only output rounding separates them)
    assert abs(con.item() - oracle["loss"].item()) < ctol * abs(oracle["loss"].item())
    otol = 1e-5 if fp32 else 4e-3          # bf16 outputs: one rounding of each gradient element
    assert rel_err(qd.grad.double().cpu(), oracle["dq"]) < otol
    assert rel_err(vd.grad.double().cpu(), oracle["dv"]) < otol
    assert abs(m.temperature.grad.item() - oracle["dT"].item()) < 1e-5 * scale

    # (5) statistics dictionary: same keys as the reference, values within tolerance
    keys = [str(k) for k in gold["stats_keys"]]
    assert sorted(stats.keys()) == keys
    sc = max(abs(float(x)) for x in gold["stats_vals"])
    stol = 1e-2 if (case.dtype == "bf16" and case.kind == "av") else 1e-4
    for k, ref in zip(keys, gold["stats_vals"]):
        assert abs(stats[k] - float(ref)) <= stol * sc, k


def _near_tie_report(q, v, T, idx_a, idx_b):
    """For argmax disagreements between two accumulation orders, check each is a genuine
    near-tie: the exact (fp64) similarities of the two candidates differ by < 2 bf16 ulps."""
    bad = (idx_a != idx_b).nonzero()
    worst = 0.0
    for i, j, a in bad.tolist():
        s = (q[i, a].double() @ v[j].double().t()) * T
        x, y = s[idx_a[i, j, a]].item(), s[idx_b[i, j, a]].item()
        worst = max(worst, abs(x - y) / max(abs(x), 1e-30))
    return len(bad), worst


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
@pytest.mark.parametrize("chunk_bytes,fused", [(None, True), (1 << 14, True), (None, False)])
def test_golden_total_loss_with_regularisers(case, chunk_bytes, fused, monkeypatch):
    """SURVEY §8(f1): total loss, regulariser values and the gradients of the TOTAL loss (dense
    non-negative pressure + positive-pair terms on top of the contrastive part) vs the reference."""
    from triad_b200 import regularizers as R
    monkeypatch.setattr(R, "USE_FUSED", fused)        # tcgen05 forward writing N vs library GEMM + elementwise kernel
    if chunk_bytes is not None:                       # many small image chunks: exercises the chunk loop
        monkeypatch.setattr(R, "CHUNK_BYTES", chunk_bytes)
    gold = load_golden(case.name)
    q, v, mask, T = build_inputs(case)
    m = _model(T, regularizers=True)
    qd, vd = q.cuda().requires_grad_(), v.cuda().requires_grad_()
    if case.kind == "av":
        clip, tok = m.compute_all_similarities_av(qd, vd)
        total, con, reg, smooth, stats = m.compute_contrastive_loss_av(clip, tok)
        assert abs(smooth.item() - float(gold["smooth"])) <= 1e-2 * abs(float(gold["smooth"])) + 1e-9
    else:
        clip, tok = m.compute_all_similarities_tv(qd, vd, mask.cuda())
        total, stats = m.compute_contrastive_loss_tv(clip, tok)
        con = m._loss_head(clip, tok, "tv", False)[0]
        reg = total - con
    fp32 = case.dtype == "fp32"
    tol = 1e-4 if fp32 else 1e-2
    assert abs(total.item() - float(gold["total"])) <= tol * abs(float(gold["total"]))
    assert abs(reg.item() - float(gold["reg"])) <= tol * abs(float(gold["reg"])) + (1e-7 if fp32 else 1e-5)
    total.backward()
    P = projection(case)
    dq = qd.grad.double().cpu() @ P if P is not None else qd.grad.double().cpu()
    dv = vd.grad.double().cpu() @ P if P is not None else vd.grad.double().cpu()
    assert rel_err(dq, gold["dq_total"]) < tol
    assert rel_err(dv, gold["dv_total"]) < tol
    # dT is a cancelling sum (sum_ij g*clip/T): tolerance relative to the sum of magnitudes, as in test_golden_parity
    oracle = O.contrastive_step_closed_form(q, v, T, mask)
    scale = (oracle["g"].abs() * oracle["clip"].abs().double()).sum().item() / T
    assert abs(m.temperature.grad.item() - float(gold["dT_total"])) < (1e-4 if fp32 else 2e-2) * scale
    # the regularisers alone: the dense part must be right on its own, not just hidden under the (much
    # larger) contrastive gradient.  Reference for this check: fp64 autograd of the oracle's restatement
    # (pinned to the reference's `reg` by tests/test_oracle_golden.py) on the same inputs.
    q64, v64 = q.double().requires_grad_(), v.double().requires_grad_()
    T64 = torch.tensor(float(T), dtype=torch.float64, requires_grad=True)
    tok64 = torch.einsum("iad,jpd->ijap", q64, v64) * T64
    reg64 = O.regularization_av(tok64, T64)[0] if case.kind == "av" else O.regularization_tv(tok64, 0.80, 0.01)
    reg64.backward()
    qd.grad = vd.grad = m.temperature.grad = None
    clip2, tok2 = (m.compute_all_similarities_av(qd, vd) if case.kind == "av"
                   else m.compute_all_similarities_tv(qd, vd, mask.cuda()))
    reg2 = (m.compute_regularization_losses_av(tok2)[0] if case.kind == "av" else m.compute_regularization_losses_tv(tok2))
    reg2.backward()
    rtol = 1e-4 if fp32 else 1e-2
    assert abs(reg2.item() - reg64.item()) <= rtol * abs(reg64.item())
    assert rel_err(qd.grad.double().cpu(), q64.grad) < rtol
    assert rel_err(vd.grad.double().cpu(), v64.grad) < rtol
    assert abs(m.temperature.grad.item() - T64.grad.item()) <= rtol * abs(T64.grad.item()) + 1e-9


@pytest.mark.parametrize("fused", [True, False])
def test_nonneg_pressure_reaches_the_clamp_floor(fused, monkeypatch):
    """Similarities below the clamp floor (lo = -20): the value clamps there and the gradient is gated off
    (torch.clamp's backward).  The fused tcgen05 path detects such tiles by their row minimum and redoes them
    with the reference's rounding; the library-GEMM path applies the gate per element."""
    from triad_b200 import regularizers as R
    monkeypatch.setattr(R, "USE_FUSED", fused)
    B, Nq, Nv, D, T, lo = 6, 40, 64, 64, 1.5, -20.0
    g = torch.Generator().manual_seed(5)
    q = (torch.randn(B, Nq, D, generator=g) * 1.2).bfloat16()
    v = (torch.randn(B, Nv, D, generator=g) * 1.2).bfloat16()
    q64, v64 = q.double().requires_grad_(), v.double().requires_grad_()
    T64 = torch.tensor(T, dtype=torch.float64, requires_grad=True)
    tok = torch.einsum("iad,jpd->ijap", q64, v64) * T64
    assert (tok < lo).float().mean().item() > 0.01           # the floor is really reached
    ref = tok.clamp(min=lo, max=0).pow(2).mean()
    ref.backward()
    qd, vd = q.cuda().requires_grad_(), v.cuda().requires_grad_()
    Td = torch.nn.Parameter(torch.tensor(T, device="cuda"))
    val = R.nonneg_pressure(qd, vd, Td, lo)
    val.backward()
    assert abs(val.item() - ref.item()) <= 1e-2 * ref.item()
    # Both paths round S to bf16 twice near the floor, exactly like the reference under autocast (model.py:387): at
    # |S| ~ 20 a bf16 ulp is 0.125, similarities within an ulp of the floor fall on either side of the gradient
    # gate, and they are the largest terms — the reference's own bf16 graph is ~9 % away from fp64 here.  So the
    # gradients are checked against that graph (ATen, bf16, materialised; small shape), and only loosely against fp64.
    qb, vb = q.cuda().requires_grad_(), v.cuda().requires_grad_()
    Tb = torch.nn.Parameter(torch.tensor(T, device="cuda"))
    tb = torch.matmul(qb.unsqueeze(1).expand(-1, B, -1, -1), vb.unsqueeze(0).expand(B, -1, -1, -1).transpose(2, 3)) * Tb
    torch.mean(torch.clamp(tb, min=lo, max=0) ** 2).backward()
    assert rel_err(qd.grad.double().cpu(), qb.grad.double().cpu()) < 1e-2
    assert rel_err(vd.grad.double().cpu(), vb.grad.double().cpu()) < 1e-2
    assert abs(Td.grad.item() - Tb.grad.item()) <= 2e-2 * abs(Tb.grad.item())
    assert rel_err(qd.grad.double().cpu(), q64.grad) < 0.15 and rel_err(vd.grad.double().cpu(), v64.grad) < 0.15


@pytest.mark.parametrize("flags", [0, FWD_1CTA, FWD_SYNC, FWD_SYNC | FWD_1CTA])
def test_tensor_core_vs_oracle_mid_size(flags):
    """B=24 x 250 x 256 x 512: tcgen05 argmax vs the CPU oracle.  Different fp32 accumulation
    orders can flip a bf16 rounding on an exact-to-the-ulp tie; every disagreement must be such
    a near-tie and they must be rare."""
    from triad_b200 import ops
    B, Nq, Nv, D = 24, 250, 256, 512
    q, v, _ = O.make_inputs(B, Nq, Nv, D, torch.bfloat16, seed=77)
    ref = O.maxmean_forward(q, v, 1.5)
    scale = ops.row_scale(None, B, Nq, torch.device("cuda"))
    Tt = torch.tensor(1.5, device="cuda")
    clip, idx = ops.maxmean_fwd(q.cuda(), v.cuda(), scale, Tt, flags=flags, check_watchdog=True)
    idx = ops.idx_to_reference_layout(idx, B, Nq).cpu()
    n_bad, worst = _near_tie_report(q, v, 1.5, idx, ref["idx"])
    assert n_bad <= 1e-4 * idx.numel(), n_bad
    assert worst < 2 ** -7, worst
    assert rel_err(clip.cpu(), ref["clip"]) < 5e-5


def test_full_size_properties_cfg2():
    """BASELINE cfg 2 (B=256, 250 frames x 256 patches, D=512, bf16) — properties that do not
    need the (16.8 GB) dense tensor."""
    from triad_b200 import ops
    B, Nq, Nv, D = 256, 250, 256, 512
    q, v, _ = O.make_inputs(B, Nq, Nv, D, torch.bfloat16, seed=1234)
    qd, vd = q.cuda(), v.cuda()
    dev = qd.device
    scale = ops.row_scale(None, B, Nq, dev)
    Tt = torch.tensor(1.5, device=dev)
    clip, idx = ops.maxmean_fwd(qd, vd, scale, Tt, check_watchdog=True)

    # (a) run-to-run determinism, bit for bit
    clip2, idx2 = ops.maxmean_fwd(qd, vd, scale, Tt)
    assert torch.equal(clip, clip2)
    assert torch.equal(ops.idx_to_reference_layout(idx, B, Nq), ops.idx_to_reference_layout(idx2, B, Nq))

    # (b) tiling independence: a sub-batch of queries against a sub-set of images reproduces the
    #     corresponding block: argmax bit-exactly (same arithmetic per element whatever the tile
    #     schedule), clip up to the fp32 summation order of the per-group partial sums
    qi, vj = slice(37, 37 + 19), slice(101, 101 + 50)
    sub_scale = ops.row_scale(None, 19, Nq, dev)
    clip_s, idx_s = ops.maxmean_fwd(qd[qi].contiguous(), vd[vj].contiguous(), sub_scale, Tt)
    assert torch.allclose(clip_s, clip[qi, vj], rtol=2e-6, atol=0)
    idx_ref = ops.idx_to_reference_layout(idx, B, Nq)            # (Bq,Bv,Nq)
    assert torch.equal(ops.idx_to_reference_layout(idx_s, 19, Nq), idx_ref[qi, vj])

    # (c) a slice against the CPU oracle (argmax bit-exact up to certified near-ties)
    ref = O.maxmean_forward(q[:6], v, 1.5)
    got = idx_ref[:6].cpu()
    n_bad, worst = _near_tie_report(q[:6], v, 1.5, got, ref["idx"])
    assert n_bad <= 1e-4 * got.numel() and worst < 2 ** -7
    assert rel_err(clip[:6].cpu(), ref["clip"]) < 5e-5

    # (d) permutation equivariance: permuting the images permutes clip columns exactly
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(3)).cuda()
    clip_p, _ = ops.maxmean_fwd(qd, vd[perm].contiguous(), scale, Tt)
    assert torch.equal(clip_p, clip[:, perm])

    # (e) loss + closed-form gradient identities: rows/cols of g sum to ~0 around the diagonal term
    row_lse, col_part = ops.infonce_partial(clip, B, 0)
    g, sums = ops.infonce_finish(clip, B, 0, row_lse, col_part.reshape(1, 2, B))
    nce = O.infonce(clip.cpu())
    assert abs(sums[0].item() / (2 * B) - nce["loss"].item()) < 1e-6 * nce["loss"].item()
    assert rel_err(g.cpu(), nce["g"]) < 1e-5
    assert g.double().sum().abs().item() < 1e-7          # sum(P) = sum(Q) = B, so sum(g) = (B + B - 2B)/(2B) = 0

    # (f) backward: linear in g (exactly, for power-of-two scaling), and checked against the oracle
    #     on a slice of queries / images
    dq, dv, dT = ops.maxmean_bwd(qd, vd, idx, g, clip, scale, Tt)
    dq2, dv2, dT2 = ops.maxmean_bwd(qd, vd, idx, g * 2, clip, scale, Tt)
    assert torch.equal(dq2.float(), dq.float() * 2) and torch.equal(dv2.float(), dv.float() * 2)
    # independent fp64 evaluation of the gather / scatter formulas with plain torch indexing (test-only)
    g64, q64, v64 = g.double(), qd.double().view(B * Nq, D), vd.double().view(B * Nv, D)
    idx_l = idx_ref.permute(1, 0, 2).reshape(B, B * Nq)           # [Bv, M]
    for i in (0, 100, 255):
        rows = torch.arange(i * Nq, (i + 1) * Nq, device=dev)
        flat = idx_l[:, rows] + (torch.arange(B, device=dev) * Nv)[:, None]          # (Bv,Nq)
        want = 1.5 * scale[rows].double()[:, None] * (g64[i][:, None, None] * v64[flat]).sum(dim=0)
        assert rel_err(dq[i].cpu(), want.cpu()) < 4e-3
    w_rows = 1.5 * scale.double()[None, :] * g64.t().repeat_interleave(Nq, dim=1)      # [Bv, M]
    for j in (0, 77, 255):
        want = torch.zeros(Nv, D, dtype=torch.float64, device=dev)
        want.index_add_(0, idx_l[j], w_rows[j][:, None] * q64)
        assert rel_err(dv[j].cpu(), want.cpu()) < 4e-3
    ssum = (g.abs() * clip.abs()).double().sum().item() / 1.5
    assert abs(dT.item() - ((g64 * clip.double()).sum() / 1.5).item()) < 1e-5 * ssum


@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("Nv", [200, 600, 2048, 3072])
def test_backward_variants_agree(Nv, masked):
    """Every backward kernel variant (dq: shared-memory pipeline for Nv <= 256, L1-resident tile for Nv > 256,
    generic L2 gather; single-block and multi-block dv, fp32-partial and bf16 dv) against the oracle's closed
    form and against each other.  Nv = 2048 and 3072 take the global dv sort with the packed bf16 gather; 3072 is
    the largest Nv the dv pass handles."""
    from triad_b200 import _lib, ops
    B, Nq, D = 20, 77, 256
    q, v, mask = O.make_inputs(B, Nq, Nv, D, torch.bfloat16, seed=41, masked=masked, min_len=3)
    ref = O.contrastive_step_closed_form(q, v, 1.5, mask)
    qd, vd = q.cuda(), v.cuda()
    scale = ops.row_scale(None if mask is None else mask.cuda(), B, Nq, qd.device)
    Tt = torch.tensor(1.5, device=qd.device)
    clip, idx = ops.maxmean_fwd(qd, vd, scale, Tt)
    g = ref["g"].float().cuda()
    # closed-form gradients for the winners the GPU actually chose (a near-tie flip, see
    # _near_tie_report, would otherwise dominate the fp32 comparison)
    idx_ref_layout = ops.idx_to_reference_layout(idx, B, Nq).cpu()
    rdq, rdv, _ = O.maxmean_backward(q, v, idx_ref_layout, g.cpu(), 1.5, ref["row_scale"], clip.cpu())
    ref = {"dq": rdq, "dv": rdv}
    outs = {}
    for name, flags, f32 in (("default", 0, False), ("dq_generic", _lib.BWD_GENERIC_DQ, False),
                             ("dq_packed", _lib.BWD_PACK_ROWS, False),
                             ("dv_generic", _lib.BWD_GENERIC_DV, False),
                             ("dv_blocks", _lib.BWD_SMALL_BLOCKS, False),
                             ("dv_blocks_generic", _lib.BWD_SMALL_BLOCKS | _lib.BWD_GENERIC_DV, False),
                             ("dv_blocks_f32", _lib.BWD_SMALL_BLOCKS, True), ("dv_f32", 0, True)):
        dq, dv, dT = ops.maxmean_bwd(qd, vd, idx, g, clip, scale, Tt, dv_f32=f32, flags=flags)
        outs[name] = (dq, dv)
        assert rel_err(dq.cpu(), ref["dq"]) < 4e-3, name
        assert rel_err(dv.cpu(), ref["dv"]) < (1e-5 if f32 else 4e-3), name
    for name in ("dq_generic", "dq_packed"):                  # same summation order: bit-identical
        assert torch.equal(outs[name][0], outs["default"][0]), name
    assert torch.equal(outs["dv_generic"][1], outs["default"][1])             # grouped vs global sort: same lists
    assert torch.equal(outs["dv_blocks_generic"][1], outs["dv_blocks"][1])
    assert torch.equal(outs["dv_f32"][1].to(torch.bfloat16), outs["default"][1])
    if masked:                                                   # padded tokens: exactly zero gradient
        assert outs["default"][0][mask.cuda() == 0].abs().max().item() == 0.0


@pytest.mark.parametrize("flags", [0, FWD_1CTA, FWD_SIMT, FWD_SYNC])
@pytest.mark.parametrize("Nv", [257, 600, 1024])
def test_more_than_256_patches(flags, Nv):
    """High-resolution galleries (cfg 5: 1024 patches per image): the tcgen05 kernel walks an image as
    256-patch sub-tiles with a running (rounded max, first argmax) per row; indices are uint16.  Ties
    between sub-tiles (duplicated patches) must resolve to the first index."""
    from triad_b200 import ops
    B, Nq, D = 5, 70, 128
    q, v, _ = O.make_inputs(B, Nq, Nv, D, torch.bfloat16, seed=90 + Nv)
    v[:, Nv - 3] = v[:, 1]            # exact duplicates in different sub-tiles -> exact ties
    v[:, 300 % Nv] = v[:, 7]
    ref = O.contrastive_step_closed_form(q, v, 1.5)
    m = _model(1.5, flags)
    qd, vd = q.cuda().requires_grad_(), v.cuda().requires_grad_()
    clip, tok = m.compute_all_similarities_av(qd, vd)
    assert tok.idx_t.dtype == torch.uint16
    con = m.compute_contrastive_loss_av(clip, tok)[1]
    con.backward()
    n_bad, worst = _near_tie_report(q, v, 1.5, tok.argmax().cpu(), ref["idx"])
    assert n_bad <= 2 and worst < 2 ** -7
    assert rel_err(tok.clip.detach().cpu(), ref["clip"]) < 5e-5
    assert abs(con.item() - ref["loss"].item()) < 1e-5 * ref["loss"].item()
    assert rel_err(qd.grad.cpu(), ref["dq"]) < 4e-3 and rel_err(vd.grad.cpu(), ref["dv"]) < 4e-3


@pytest.mark.parametrize("pack", [True, False])
@pytest.mark.parametrize("holes", [False, True])
def test_masked_text_shape_cfg3_slice(pack, holes):
    """cfg 3 flavour: 77 text tokens with ragged right-padded masks (n_i in [8,77]).  pack: zero-weight
    rows are dropped before the GEMM (the default for bf16) vs. computed and multiplied by 0; both must give
    the same clip / loss / gradients.  holes: masks that are not prefixes (zeros in the middle, an all-zero
    caption) — the packing is by weight, not by length."""
    B, Nq, Nv, D = 48, 77, 256, 512
    q, v, mask = O.make_inputs(B, Nq, Nv, D, torch.bfloat16, seed=31, masked=True, min_len=8)
    if holes:
        mask[3, 2:5] = 0
        mask[7, 0] = 0
        mask[11] = 0                    # clamp(sum,1e-7) branch of model.py:511: clip row of zeros
    m = _model(1.5)
    m.triad_pack_masked_rows = pack
    qd, vd = q.cuda().requires_grad_(), v.cuda().requires_grad_()
    clip, tok = m.compute_all_similarities_tv(qd, vd, mask.cuda())
    loss, stats = m.compute_contrastive_loss_tv(clip, tok)
    loss.backward()
    ref = O.contrastive_step_closed_form(q, v, 1.5, mask)
    n_bad, worst = _near_tie_report(q, v, 1.5, tok.argmax().cpu(), ref["idx"])
    assert n_bad <= 1e-4 * ref["idx"].numel() and worst < 2 ** -7
    assert rel_err(tok.clip.detach().cpu(), ref["clip"]) < 5e-5      # see ctol in test_golden_parity
    assert abs(loss.item() - ref["loss"].item()) < 1e-5 * ref["loss"].item()
    assert rel_err(qd.grad.cpu(), ref["dq"]) < 4e-3 and rel_err(vd.grad.cpu(), ref["dv"]) < 4e-3
    # padded tokens receive exactly zero gradient (mask multiplies their maxima by 0, model.py:510)
    assert qd.grad[mask.cuda() == 0].abs().max().item() == 0.0
    assert tok.packed == pack
    if pack:       # the winners recorded by the packed forward are the full forward's, on every kept row
        from triad_b200 import ops
        kept = mask.bool()[:, None, :].expand(B, B, Nq)
        got = ops.idx_to_reference_layout(tok.idx_t, B, Nq).cpu()
        assert torch.equal(got[kept], tok.argmax().cpu()[kept])


def test_dv_many_row_groups():
    """More than 32 sort groups per query block (narrow D, many rows): the grouped dv gather refills its
    lane-resident segment table; result must equal the global-sort path bit for bit."""
    from triad_b200 import _lib, ops
    Bq, Bv, Nq, Nv, D = 1100, 4, 250, 32, 64          # 275 000 rows = 34 groups of 8192
    g = torch.Generator(device="cuda").manual_seed(3)
    q = (torch.randn(Bq, Nq, D, generator=g, device="cuda") / D ** 0.5).bfloat16()
    v = (torch.randn(Bv, Nv, D, generator=g, device="cuda") / D ** 0.5).bfloat16()
    scale = ops.row_scale(None, Bq, Nq, q.device)
    Tt = torch.tensor(1.5, device="cuda")
    clip, idx = ops.maxmean_fwd(q, v, scale, Tt)
    gw = torch.randn(Bq, Bv, generator=g, device="cuda")
    _, dv_a, _ = ops.maxmean_bwd(q, v, idx, gw, clip, scale, Tt, need_dq=False, need_dT=False, dv_f32=True)
    _, dv_b, _ = ops.maxmean_bwd(q, v, idx, gw, clip, scale, Tt, need_dq=False, need_dT=False, dv_f32=True,
                                 flags=_lib.BWD_GENERIC_DV)
    assert torch.equal(dv_a, dv_b)
    # and against a direct fp64 evaluation of the scatter
    idx_ref = ops.idx_to_reference_layout(idx, Bq, Nq)                       # (Bq,Bv,Nq)
    w = (gw.double()[:, :, None] * scale.view(Bq, 1, Nq).double() * 1.5)    # (Bq,Bv,Nq)
    ref = torch.zeros(Bv, Nv, D, dtype=torch.float64, device="cuda")
    for j in range(Bv):
        ref[j].index_add_(0, idx_ref[:, j].reshape(-1), (w[:, j].reshape(-1, 1) * q.double().view(-1, D)))
    assert rel_err(dv_a.double().cpu(), ref.cpu()) < 1e-5


@pytest.mark.parametrize("masked", [False, True])
def test_sharded_step_single_rank_cuda(masked):
    """triad_b200.dist.sharded_contrastive_step with the product (CUDA) kernels on one rank — the code every
    rank runs under torchrun (collectives are identity at world size 1; the gloo tests cover them)."""
    from triad_b200.dist import sharded_contrastive_step
    B, Nq, Nv, D = 12, 40, 96, 128
    q, v, mask = O.make_inputs(B, Nq, Nv, D, torch.bfloat16, seed=51, masked=masked, min_len=2)
    ref = O.contrastive_step_closed_form(q, v, 1.5, mask)
    out = sharded_contrastive_step(q.cuda(), v.cuda(), torch.tensor(1.5, device="cuda"),
                                   mask.cuda() if masked else None)
    assert abs(out["loss"].item() - ref["loss"].item()) < 1e-5 * ref["loss"].item()
    assert rel_err(out["dq"].cpu(), ref["dq"]) < 4e-3 and rel_err(out["dv"].cpu(), ref["dv"]) < 4e-3
    assert abs(out["dT"].item() - ref["dT"].item()) < 1e-4 * (ref["g"].abs() * ref["clip"].abs().double()).sum().item()


@pytest.mark.parametrize("kind", ["av", "tv"])
def test_sharded_regulariser_step_single_rank_cuda(kind):
    """triad_b200.dist.sharded_regularizer_step with the product kernels on one rank vs fp64 autograd of the oracle's
    restatement (the 2-rank collectives are covered by the gloo tests)."""
    from triad_b200.dist import sharded_regularizer_step
    B, Nq, Nv, D, T = 8, 24, 64, 128, 0.9
    q, v, _ = O.make_inputs(B, Nq, Nv, D, torch.bfloat16, seed=71)
    q, v = (q.float() * 3).bfloat16(), (v.float() * 3).bfloat16()
    q64, v64 = q.double().requires_grad_(), v.double().requires_grad_()
    T64 = torch.tensor(T, dtype=torch.float64, requires_grad=True)
    tok = torch.einsum("iad,jpd->ijap", q64, v64) * T64
    reg = O.regularization_av(tok, T64)[0] if kind == "av" else O.regularization_tv(tok, 0.01, 0.5)
    reg.backward()
    out = sharded_regularizer_step(q.cuda(), v.cuda(), torch.tensor(T, device="cuda"), kind,
                                   patch_sparsity_threshold=0.01, patch_sparsity_weight=0.5)
    assert abs(out["reg"].item() - reg.item()) <= 1e-2 * abs(reg.item())
    assert rel_err(out["dq"].double().cpu(), q64.grad) < 1e-2
    assert rel_err(out["dv"].double().cpu(), v64.grad) < 1e-2
    assert abs(out["dT"].item() - T64.grad.item()) <= 1e-2 * abs(T64.grad.item())


def test_two_modalities_one_backward_and_no_grad_eval():
    """train.py computes an audio-visual and a text-visual loss in the same iteration and back-propagates their
    sum: the second forward must not disturb anything the first one's backward needs (shared workspaces); and the
    whole loss (with regularisers) evaluates under torch.no_grad() without building gradients."""
    B, Na, Nt, Nv, D = 6, 40, 16, 64, 128
    a, v, _ = O.make_inputs(B, Na, Nv, D, torch.bfloat16, seed=61)
    t, _, mask = O.make_inputs(B, Nt, Nv, D, torch.bfloat16, seed=62, masked=True, min_len=2)
    m = _model(1.5, regularizers=True)

    def run(which):
        ad, td, vd = a.cuda().requires_grad_(), t.cuda().requires_grad_(), v.cuda().requires_grad_()
        m.temperature.grad = None
        total = 0
        if "av" in which:
            clip, tok = m.compute_all_similarities_av(ad, vd)
            total = total + m.compute_contrastive_loss_av(clip, tok)[0]
        if "tv" in which:
            clip2, tok2 = m.compute_all_similarities_tv(td, vd, mask.cuda())
            total = total + m.compute_contrastive_loss_tv(clip2, tok2)[0]
        total.backward()
        z = lambda x: torch.zeros(1) if x is None else x.float().cpu()
        return total.item(), z(ad.grad), z(td.grad), z(vd.grad), m.temperature.grad.item()

    both, av, tv = run(("av", "tv")), run(("av",)), run(("tv",))
    assert abs(both[0] - (av[0] + tv[0])) < 1e-5 * abs(both[0])
    assert torch.equal(both[1], av[1]) and torch.equal(both[2], tv[2])           # da, dt: untouched by the other loss
    assert rel_err(both[3], av[3] + tv[3]) < 1e-2                                 # dv accumulates both (bf16 adds)
    assert abs(both[4] - (av[4] + tv[4])) < 1e-4 * max(1.0, abs(both[4]))
    with torch.no_grad():
        clip, tok = m.compute_all_similarities_av(a.cuda(), v.cuda())
        total = m.compute_contrastive_loss_av(clip, tok)[0]
    assert not total.requires_grad and abs(total.item() - av[0]) < 1e-5 * abs(av[0])


def test_retrieval_against_reference_goldens():
    from triad_b200 import retrieval as R
    gold = load_golden("retrieval")
    g = torch.Generator().manual_seed(77)
    row = 0
    for n, (nq, nv, d) in enumerate(gold["agg_shapes"].tolist()):
        qf = torch.randn(nq, d, generator=g)
        vf = torch.randn(nv, d, generator=g)
        if n != 1:
            qf = torch.nn.functional.normalize(qf, dim=1)
            vf = torch.nn.functional.normalize(vf, dim=1)
        for T in gold["agg_T"].tolist():
            ref = gold["agg_vals"][row]
            row += 1
            got = [R.aggregator_av_a2v(qf.cuda(), vf.cuda(), T), R.aggregator_av_v2a(qf.cuda(), vf.cuda(), T),
                   R.aggregator_tv_t2v(qf.cuda(), vf.cuda(), T), R.aggregator_tv_v2t(qf.cuda(), vf.cuda(), T)]
            assert np.allclose(got, ref, rtol=1e-4, atol=1e-6), (n, T, got, ref)
    rec = R.compute_recall_at_k(gold["recall_sim"])
    assert np.allclose([rec["r1"], rec["r5"], rec["r10"], rec["r20"]], gold["recall_vals"])


def test_retrieval_matrix_topk_and_simmat():
    from triad_b200 import retrieval as R
    g = torch.Generator().manual_seed(5)
    N = 12
    qs = [torch.nn.functional.normalize(torch.randn(int(n), 64, generator=g), dim=1) for n in torch.randint(3, 20, (N,), generator=g)]
    vs = [torch.nn.functional.normalize(torch.randn(40, 64, generator=g), dim=1) for _ in range(N)]
    for direction, name in ((0, "q2v"), (1, "v2q")):
        sim = R.pairwise_similarity(qs, vs, 0.7, direction).cpu()
        ref = torch.tensor([[O.aggregate_pair(qs[i], vs[j], 0.7, name) for j in range(N)] for i in range(N)])
        assert torch.allclose(sim, ref, rtol=1e-4, atol=1e-6)
    m = R.metrics_from_features(qs, vs, 0.7, "cuda", "av")
    assert sorted(m) == sorted([f"{a}_r{k}" for a in ("A->V", "V->A") for k in (1, 5, 10, 20)])
    # top-k over a bf16 gallery (cfg 5 flavour, small): ids and scores vs torch.topk of the oracle scores
    q = torch.nn.functional.normalize(torch.randn(77, 512, generator=g), dim=1).bfloat16()
    gal = torch.nn.functional.normalize(torch.randn(300, 256, 512, generator=g), dim=2).bfloat16()
    s, ids = R.retrieve_topk(q.cuda(), gal.cuda(), 1.5, 10)
    scores = R._scores(q.cuda(), gal.cuda(), 1.5, 0)
    ts, ti = torch.topk(scores, 10)
    assert torch.equal(ids.long(), ti) and torch.equal(s, ts)
    ref0 = O.aggregate_pair(q.float(), gal[int(ids[0])].float(), 1.5, "q2v")
    assert abs(s[0].item() - ref0) < 1e-2 * abs(ref0)
    # compute_similarity_matrix
    gold = load_golden("retrieval")
    g2 = torch.Generator().manual_seed(77)
    for (nq, nv, d) in gold["agg_shapes"].tolist():
        torch.randn(nq, d, generator=g2); torch.randn(nv, d, generator=g2)
    torch.randn(60, 60, generator=g2)
    f1 = torch.randn(3, 9, 32, generator=g2)
    f2 = torch.randn(3, 17, 32, generator=g2)
    out = _model(1.5).compute_similarity_matrix(f1.cuda(), f2.cuda()).cpu().numpy()
    assert np.allclose(out, gold["simmat"], atol=1e-5)


def test_errors_are_loud():
    from triad_b200 import ops
    from triad_b200._lib import TriadError
    m = _model(1.5)
    with pytest.raises(RuntimeError):
        m.compute_all_similarities_av(torch.randn(2, 3, 64), torch.randn(2, 5, 64))       # CPU tensors
    with pytest.raises(TypeError):
        m.compute_all_similarities_av(torch.randn(2, 3, 64).cuda().half(), torch.randn(2, 5, 64).cuda().half())
    with pytest.raises(TriadError):
        m.compute_all_similarities_av(torch.randn(2, 3, 60).cuda(), torch.randn(2, 5, 60).cuda())  # D % 8


@pytest.mark.parametrize("B", [1, 2, 7, 33, 256, 600])
def test_fused_head_matches_the_block_kernels(B):
    """triad_contrastive_head (2 launches: InfoNCE + statistics + temperature-calibration term) against the
    partial/finish pair the sharded path uses (same math; the column partials are combined over different row blocks,
    so equal to fp32 rounding, not bit for bit), and its scalars against the reference's (model.py:420-427, :453-459)."""
    from triad_b200 import ops
    gen = torch.Generator().manual_seed(B)
    clip = (torch.randn(B, B, generator=gen) * 2).cuda()
    for T in (1.5, 0.8):
        Tt = torch.tensor(T, device="cuda")
        g, sums, out = ops.contrastive_head(clip, Tt)
        row_lse, col_part = ops.infonce_partial(clip, B, 0)
        g2, sums2 = ops.infonce_finish(clip, B, 0, row_lse, col_part.reshape(1, 2, B))
        assert torch.allclose(g, g2, rtol=1e-5, atol=1e-9)
        assert torch.allclose(sums[:7], sums2[:7], rtol=1e-6, atol=1e-9)
        assert rel_err(g.cpu(), O.infonce(clip.cpu())["g"]) < 1e-5
        nce = O.infonce(clip.cpu())
        assert abs(out[0].item() - nce["loss"].item()) <= 1e-6 * abs(nce["loss"].item())
        T64 = torch.tensor(T, dtype=torch.float64, requires_grad=True)
        cal = 20.0 * torch.clamp(-torch.log(T64), min=0) ** 2
        cal.backward()
        assert abs(out[1].item() - cal.item()) <= 1e-6 * max(cal.item(), 1e-30)
        assert abs(out[2].item() - (out[0].item() + out[1].item())) <= 1e-6 * abs(out[2].item())
        assert abs(out[3].item() - T64.grad.item()) <= 1e-6 * max(abs(T64.grad.item()), 1e-30)
    g, sums, out = ops.contrastive_head(clip, None)
    assert out[1].item() == 0.0 and out[3].item() == 0.0


def test_loss_uses_the_clip_sims_argument():
    """compute_contrastive_loss_* compute the loss from the clip_sims ARGUMENT (model.py:430, :544): the matrix the
    similarity call returned maps to the handle's fp32 copy, an edited one is honoured as given."""
    B, Nq, Nv, D = 6, 20, 64, 64
    q, v, _ = O.make_inputs(B, Nq, Nv, D, torch.bfloat16, seed=3)
    m = _model(1.5)
    qd, vd = q.cuda().requires_grad_(), v.cuda().requires_grad_()
    clip, tok = m.compute_all_similarities_av(qd, vd)
    base = m.compute_contrastive_loss_av(clip, tok)[1]
    edited = clip.float() * 0.5
    con = m.compute_contrastive_loss_av(edited, tok)[1]
    want = O.infonce(edited.detach().cpu())["loss"]
    assert abs(con.item() - want.item()) <= 1e-5 * abs(want.item())
    assert abs(con.item() - base.item()) > 1e-3                      # really a different loss
    con.backward()                                                   # gradients flow through the edit
    ref = O.contrastive_step_closed_form(q, v, 1.5)
    g_half = O.infonce(edited.detach().cpu())["g"] * 0.5
    dq, dv, _ = O.maxmean_backward(q, v, ref["idx"], g_half.float(), 1.5, ref["row_scale"], ref["clip"])
    assert rel_err(qd.grad.double().cpu(), dq) < 1e-2 and rel_err(vd.grad.double().cpu(), dv) < 1e-2


def test_stats_mapping_behaves_like_the_reference_dict():
    import copy
    import json
    import pickle
    q, v, _ = O.make_inputs(4, 10, 32, 64, torch.bfloat16, seed=9)
    m = _model(1.5)
    clip, tok = m.compute_all_similarities_av(q.cuda(), v.cuda())
    stats = m.compute_contrastive_loss_av(clip, tok)[4]
    d = {}
    d.update(stats)                                                  # train.py:1080
    assert sorted(d) == sorted(stats.keys()) and len(d) == 6
    assert all(k in stats for k in d) and {**stats} == d
    assert json.loads(json.dumps(stats.to_dict())) == d
    assert pickle.loads(pickle.dumps(stats)) == d and copy.deepcopy(stats) == d


# ---- round 2: argmax pinned against the reference's CUDA path, with the flip count reported -------------------------
def _report(name, payload):
    """Parity counts are printed and, when the scratch directory exists, appended to gpurun_out/parity_counts.jsonl."""
    import json
    import os
    line = json.dumps({"test": name, **payload})
    print(line)
    out = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    if os.path.isdir(out):
        with open(os.path.join(out, "parity_counts.jsonl"), "a") as f:
            f.write(line + "\n")


def test_argmax_flip_count_vs_reference_cuda_path():
    """The deployment path of the reference is torch-CUDA eager (cuBLAS bf16 matmul, src/model.py:384-391 under
    train.py:76).  B=32 x 250 x 256 x 512 bf16: winners of the fused kernel vs (a) the reference's OWN methods run on
    this GPU (oracle/_ref staged copy; the oracle's restatement on CUDA if it is absent) and (b) the CPU oracle.
    Disagreements can only be accumulation-order flips of a bf16 rounding on an exact-to-the-ulp tie: counted,
    bounded, and each certified."""
    from oracle import ref_loader
    from triad_b200 import ops
    B, Nq, Nv, D, T = 32, 250, 256, 512, 1.5
    q, v, _ = O.make_inputs(B, Nq, Nv, D, torch.bfloat16, seed=2024)
    qd, vd = q.cuda(), v.cuda()
    scale = ops.row_scale(None, B, Nq, qd.device)
    Tt = torch.tensor(T, device="cuda")
    clip, idx = ops.maxmean_fwd(qd, vd, scale, Tt, check_watchdog=True)
    got = ops.idx_to_reference_layout(idx, B, Nq)                      # (B,B,Nq) on the GPU

    ref = ref_loader.load()
    with torch.no_grad():
        if ref is not None:
            M = ref[0].MultiModalModel
            stub = ref_loader.make_stub(M, T, regularizers=False, device="cuda")
            clip_ref, tok_ref = M.compute_all_similarities_av(stub, qd, vd)
            src = "reference (oracle/_ref/model.py) on CUDA"
        else:
            tok_ref = torch.matmul(qd[:, None].expand(B, B, Nq, D), vd[None].expand(B, B, Nv, D).transpose(2, 3)) * Tt
            clip_ref = tok_ref.max(dim=3).values.mean(dim=2)
            src = "restatement of model.py:384-391 on CUDA (oracle/_ref not staged)"
        assert tok_ref.dtype == torch.bfloat16 and clip_ref.dtype == torch.bfloat16
        idx_cuda = tok_ref.max(dim=3).indices
    n_cuda, worst_cuda = certify_near_ties(qd, vd, got, idx_cuda)
    cpu = O.maxmean_forward(q, v, T)
    n_cpu, worst_cpu = certify_near_ties(qd, vd, got, cpu["idx"].cuda())
    n_ref_vs_cpu = int((idx_cuda.cpu() != cpu["idx"]).sum())           # the two reference paths disagree with each other too
    numel = got.numel()
    _report("argmax_flip_count", {"rows": numel, "vs": src, "mismatch_vs_reference_cuda": n_cuda,
                                  "mismatch_vs_cpu_oracle": n_cpu, "reference_cuda_vs_cpu": n_ref_vs_cpu,
                                  "worst_gap_bf16_ulps": max(worst_cuda, worst_cpu)})
    assert n_cuda <= max(2, 1e-4 * numel) and n_cpu <= max(2, 1e-4 * numel), (n_cuda, n_cpu)
    assert worst_cuda < 2.0 and worst_cpu < 2.0           # in bf16 ulps of the accumulator
    assert rel_err(clip.cpu(), clip_ref.float().cpu()) < 1e-2          # the reference's clip is bf16
    assert rel_err(clip.cpu(), cpu["clip"]) < 5e-5


def test_full_size_cfg3_masked():
    """BASELINE cfg 3 at its own size: B=512, 77 text tokens with ragged masks, 256 patches, D=512, bf16, through the
    drop-in methods (padded tokens packed out).  Oracle on a slice of queries (all 512 images); loss and g from the
    oracle's InfoNCE on the full clip matrix; dq on the slice, dv on three images by an fp64 evaluation."""
    from triad_b200 import ops
    B, Nq, Nv, D, T = 512, 77, 256, 512, 1.5
    q, v, mask = O.make_inputs(B, Nq, Nv, D, torch.bfloat16, seed=303, masked=True, min_len=8)
    m = _model(T)
    qd, vd, md = q.cuda().requires_grad_(), v.cuda().requires_grad_(), mask.cuda()
    clip, tok = m.compute_all_similarities_tv(qd, vd, md)
    loss, stats = m.compute_contrastive_loss_tv(clip, tok)
    loss.backward()
    assert tok.packed
    sl = [0, 1, 77, 255, 300, 511]
    ref = O.maxmean_forward(q[sl], v, T, mask[sl])
    got = tok.argmax()[sl]
    n_bad, worst = certify_near_ties(qd.detach()[sl], vd.detach(), got, ref["idx"].cuda())
    _report("cfg3_full_size", {"rows": got.numel(), "mismatch_vs_cpu_oracle": n_bad, "worst_gap_bf16_ulps": worst})
    assert n_bad <= max(2, 1e-4 * got.numel()) and worst < 2.0
    assert rel_err(tok.clip.detach()[sl].cpu(), ref["clip"]) < 5e-5
    nce = O.infonce(tok.clip.detach().cpu())
    assert abs(loss.item() - nce["loss"].item()) < 1e-5 * nce["loss"].item()
    g = nce["g"]
    rdq, _, _ = O.maxmean_backward(q[sl], v, got.cpu(), g[sl].float(), T, ref["row_scale"], ref["clip"])
    assert rel_err(qd.grad[sl].cpu(), rdq) < 4e-3
    assert qd.grad[md == 0].abs().max().item() == 0.0
    idx_l = tok.argmax().permute(1, 0, 2).reshape(B, B * Nq)                            # [Bv, M] winners (GPU)
    scale = ops.row_scale(md, B, Nq, qd.device).double()
    w_rows = T * scale[None, :] * g.cuda().t().repeat_interleave(Nq, dim=1)             # [Bv, M]
    q64 = qd.detach().double().view(B * Nq, D)
    for j in (0, 200, 511):
        want = torch.zeros(Nv, D, dtype=torch.float64, device="cuda")
        want.index_add_(0, idx_l[j], w_rows[j][:, None] * q64)
        assert rel_err(vd.grad[j].cpu(), want.cpu()) < 4e-3


def test_cfg4_rank_shape_slice():
    """BASELINE cfg 4, one rank's share at 8 GPUs: 1024 queries x 8192 images (V = 2.1 GB: the chunk-synchronous tile
    order, selected by size, not by the test flag).  Winners and clip of one query against ALL 8192 images and of eight
    queries against 64 spread images vs the CPU oracle; dq of those queries and dv of two images by fp64 evaluation."""
    from triad_b200 import ops
    Bq, Bv, Nq, Nv, D, T = 1024, 8192, 250, 256, 512, 1.5
    g0 = torch.Generator(device="cuda").manual_seed(44)
    qd = (torch.randn(Bq, Nq, D, generator=g0, device="cuda") / D ** 0.5).bfloat16()
    vd = (torch.randn(Bv, Nv, D, generator=g0, device="cuda") / D ** 0.5).bfloat16()
    scale = ops.row_scale(None, Bq, Nq, qd.device)
    Tt = torch.tensor(T, device="cuda")
    clip, idx = ops.maxmean_fwd(qd, vd, scale, Tt, check_watchdog=True)
    idx_v = idx.view(Bv, Bq, ops.nq_padded(Nq))[:, :, :Nq]                               # [Bv,Bq,Nq] view
    # (a) one query x all images
    qi = 517
    ref = O.maxmean_forward(qd[qi:qi + 1].cpu(), vd.cpu(), T)
    got = idx_v[:, qi].to(torch.int64)[None]                                             # (1,Bv,Nq)
    n1, w1 = certify_near_ties(qd[qi:qi + 1], vd, got, ref["idx"].cuda())
    assert rel_err(clip[qi:qi + 1].cpu(), ref["clip"]) < 5e-5
    # (b) eight queries x 64 spread images
    qs = [0, 1, 255, 256, 600, 777, 1000, 1023]
    js = list(range(5, Bv, 128))
    ref2 = O.maxmean_forward(qd[qs].cpu(), vd[js].cpu(), T)
    got2 = idx_v[js][:, qs].permute(1, 0, 2).to(torch.int64)
    n2, w2 = certify_near_ties(qd[qs], vd[js], got2, ref2["idx"].cuda())
    _report("cfg4_rank_shape", {"rows": got.numel() + got2.numel(), "mismatch_vs_cpu_oracle": n1 + n2,
                                "worst_gap_bf16_ulps": max(w1, w2)})
    assert n1 + n2 <= max(2, 1e-4 * (got.numel() + got2.numel())) and max(w1, w2) < 2.0
    assert rel_err(clip[qs][:, js].cpu(), ref2["clip"]) < 5e-5
    # (c) backward at this shape: dq rows of two queries and dv of two images vs fp64 evaluation of the formulas
    gw = torch.randn(Bq, Bv, generator=g0, device="cuda") / (Bq * Bv) ** 0.5
    dq, dv, dT = ops.maxmean_bwd(qd, vd, idx, gw, clip, scale, Tt)
    v64 = vd.double().view(Bv * Nv, D)
    for i in (0, 517):
        flat = idx_v[:, i].to(torch.int64) + (torch.arange(Bv, device="cuda") * Nv)[:, None]      # (Bv,Nq)
        want = torch.zeros(Nq, D, dtype=torch.float64, device="cuda")
        for j0 in range(0, Bv, 1024):                                                     # chunks: (1024,Nq,D) fp64 = 1 GB
            want += (gw[i, j0:j0 + 1024].double()[:, None, None] * v64[flat[j0:j0 + 1024]]).sum(dim=0)
        want *= T * scale[i * Nq:(i + 1) * Nq].double()[:, None]
        assert rel_err(dq[i].cpu(), want.cpu()) < 4e-3
    q64 = qd.double().view(Bq * Nq, D)
    for j in (3, 8191):
        w_rows = T * scale.double() * gw[:, j].double().repeat_interleave(Nq)
        want = torch.zeros(Nv, D, dtype=torch.float64, device="cuda")
        want.index_add_(0, idx_v[j].reshape(-1).to(torch.int64), w_rows[:, None] * q64)
        assert rel_err(dv[j].cpu(), want.cpu()) < 4e-3
    ssum = (gw.abs() * clip.abs()).double().sum().item() / T
    assert abs(dT.item() - ((gw.double() * clip.double()).sum() / T).item()) < 1e-5 * ssum


def test_tripped_watchdog_is_loud():
    """A pipeline watchdog that fires (a barrier wait that never completes) must not return a plausible-looking
    result: the forward's clip and the backward's dq come back NaN — the loss is NaN — and the status call reports
    TRIAD_ERR_TIMEOUT.  The flag is raised artificially here (test-only flags of the C ABI)."""
    from triad_b200 import _lib, ops
    q, v, mask = O.make_inputs(6, 40, 64, 128, torch.bfloat16, seed=12, masked=True, min_len=4)
    qd, vd = q.cuda(), v.cuda()
    Tt = torch.tensor(1.5, device="cuda")
    for msk, flags in ((None, 0), (mask.cuda(), _lib.FWD_PACK_ROWS)):
        scale = ops.row_scale(msk, 6, 40, qd.device)
        clip, idx = ops.maxmean_fwd(qd, vd, scale, Tt, flags=flags | _lib.FWD_TEST_TRIP_WATCHDOG)
        assert bool(torch.isnan(clip).all())
        with pytest.raises(_lib.TriadError) as e:
            ops.maxmean_fwd(qd, vd, scale, Tt, flags=flags | _lib.FWD_TEST_TRIP_WATCHDOG, check_watchdog=True)
        assert e.value.status == -8
    scale = ops.row_scale(None, 6, 40, qd.device)
    clip, idx = ops.maxmean_fwd(qd, vd, scale, Tt)
    assert bool(torch.isfinite(clip).all())
    g = torch.randn(6, 6, device="cuda")
    dq, dv, dT = ops.maxmean_bwd(qd, vd, idx, g, clip, scale, Tt, flags=_lib.BWD_TEST_TRIP_WATCHDOG)
    assert bool(torch.isnan(dq.float()).all())
    dq, dv, dT = ops.maxmean_bwd(qd, vd, idx, g, clip, scale, Tt)
    assert bool(torch.isfinite(dq.float()).all())


def test_dense_regulariser_with_patch_dropout_shapes(monkeypatch):
    """Patch dropout leaves Nv ~ 190-210 patches (model.py:296-307), not a multiple of 8: the tcgen05 dense-regulariser
    forward still takes the shape (images padded with zero patches, which contribute exactly nothing) and agrees with
    the library-GEMM path and with fp64 autograd."""
    from triad_b200 import regularizers as R
    B, Nq, Nv, D, T, lo = 5, 60, 201, 128, 1.5, -60.0
    g = torch.Generator().manual_seed(8)
    q = (torch.randn(B, Nq, D, generator=g) * 0.4).bfloat16()
    v = (torch.randn(B, Nv, D, generator=g) * 0.4).bfloat16()
    assert R.fused_supported(q.cuda(), v.cuda())
    outs = {}
    for fused in (True, False):
        monkeypatch.setattr(R, "USE_FUSED", fused)
        qd, vd = q.cuda().requires_grad_(), v.cuda().requires_grad_()
        Td = torch.nn.Parameter(torch.tensor(T, device="cuda"))
        val = R.nonneg_pressure(qd, vd, Td, lo)
        val.backward()
        outs[fused] = (val.item(), qd.grad, vd.grad, Td.grad.item())
        assert vd.grad.shape == (B, Nv, D)
    q64, v64 = q.double().requires_grad_(), v.double().requires_grad_()
    T64 = torch.tensor(T, dtype=torch.float64, requires_grad=True)
    ref = (torch.einsum("iad,jpd->ijap", q64, v64) * T64).clamp(min=lo, max=0).pow(2).mean()
    ref.backward()
    for fused in (True, False):
        val, dq, dv, dT = outs[fused]
        assert abs(val - ref.item()) <= 1e-2 * ref.item()
        assert rel_err(dq.double().cpu(), q64.grad) < 1e-2 and rel_err(dv.double().cpu(), v64.grad) < 1e-2
        assert abs(dT - T64.grad.item()) <= 1e-2 * abs(T64.grad.item())
    assert rel_err(outs[True][1], outs[False][1]) < 4e-3 and rel_err(outs[True][2], outs[False][2]) < 4e-3
