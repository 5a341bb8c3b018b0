"""GPU tier: triad_maxmean_fwd_nonneg — the max-mean forward and N = dL/d<q,v> of the dense non-negative-pressure
regulariser (src/model.py:411-412 / :525-526) from ONE pass over the similarities — against the two single-purpose
kernels it merges (bit-identical) and against a plain fp32 evaluation of the reference's formulas."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _inputs(Bq, Bv, Nq, Nv, D, seed, gain=1.0):
    g = torch.Generator().manual_seed(seed)
    q = (torch.randn(Bq, Nq, D, generator=g) * gain / D ** 0.5).bfloat16().cuda()
    v = (torch.randn(Bv, Nv, D, generator=g) * gain / D ** 0.5).bfloat16().cuda()
    return q, v


def _dense_reference(q, v, T, lo, coef):
    """N and the two sums in fp64 from the bf16-rounded similarities the reference builds (model.py:387)."""
    Bq, Nq, D = q.shape
    Bv, Nv, _ = v.shape
    raw = (q.reshape(-1, D).float() @ v.reshape(-1, D).float().t())                 # [M, Bv*Nv] exact fp32 accumulate
    S = raw.double() * T
    n = S.clamp(max=0)
    gate = (S >= lo)
    N = coef * T * torch.where(gate, n, torch.zeros_like(n))
    return N, (n.clamp(min=lo) ** 2).sum(), (coef * torch.where(gate, n, torch.zeros_like(n)) * raw.double()).sum()


SHAPES = [
    # Bq, Bv, Nq, Nv, D     (row counts that are not multiples of the 256-row tile, patch counts that clip the 64-column
    #                        store boxes, a single image, D < 512)
    (6, 6, 50, 256, 512),
    (5, 7, 77, 200, 512),
    (3, 4, 250, 72, 256),
    (9, 2, 33, 8, 64),
    (4, 5, 130, 136, 128),
    (2, 1, 300, 256, 512),
]


@pytest.mark.parametrize("shape", SHAPES, ids=["x".join(map(str, s)) for s in SHAPES])
@pytest.mark.parametrize("flags", [0, 2, 8], ids=["2cta", "1cta", "sync-chunks"])
def test_merged_forward_equals_its_parts(shape, flags):
    from triad_b200 import ops
    from triad_b200 import regularizers as R
    Bq, Bv, Nq, Nv, D = shape
    q, v = _inputs(Bq, Bv, Nq, Nv, D, 11 + Nq)
    T = torch.tensor(1.5, device="cuda")
    scale = ops.row_scale(None, Bq, Nq, q.device)
    lo, coef = -60.0, 2.0 / (float(Bq * Nq) * Bv * Nv)
    clip0, idx0 = ops.maxmean_fwd(q, v, scale, T, want_idx=True, flags=flags, check_watchdog=True)
    sums0 = torch.zeros(2, dtype=torch.float64, device="cuda")
    N0 = R.nonneg_fused_chunk(q, v, T, lo, coef, True, sums0)
    clip1, idx1, N1, sums1 = ops.maxmean_fwd_nonneg(q, v, scale, T, lo, coef, flags=flags)
    torch.cuda.synchronize()
    assert torch.equal(clip0, clip1)
    assert torch.equal(idx0.view(Bv, Bq, -1)[:, :, :Nq], idx1.view(Bv, Bq, -1)[:, :, :Nq])
    assert torch.equal(N0, N1)
    # both passes sum in the same emission warps; the regulariser-only pass always runs CTA pairs in the default tile
    # order, so with other flags the per-tile sums are added in a different order: fp32 association, nothing else
    if flags == 0:
        assert torch.equal(sums0, sums1)
    else:
        assert ((sums0 - sums1).abs() <= 1e-6 * sums0.abs()).all()
    Nref, s2, sT = _dense_reference(q, v, 1.5, lo, coef)
    err = ((N1.double() - Nref).norm() / Nref.norm()).item()
    assert err < 4e-3, err                                                          # one bf16 rounding of N
    assert abs(sums1[0].item() - s2.item()) <= 1e-5 * abs(s2.item())
    assert abs(sums1[1].item() - sT.item()) <= 1e-5 * abs(sT.item())


def test_merged_forward_at_the_clamp_floor():
    """Similarities below lo: the tile is redone with the reference's rounding and the gradient gate; the merged kernel
    and the regulariser-only kernel take the same exact path."""
    from triad_b200 import ops
    from triad_b200 import regularizers as R
    Bq, Bv, Nq, Nv, D = 6, 6, 40, 64, 64
    q, v = _inputs(Bq, Bv, Nq, Nv, D, 5, gain=1.2 * 8.0)
    T = torch.tensor(1.5, device="cuda")
    lo, coef = -20.0, 2.0 / (float(Bq * Nq) * Bv * Nv)
    raw = q.reshape(-1, D).float() @ v.reshape(-1, D).float().t()
    assert ((raw * 1.5) < lo).float().mean().item() > 0.01
    scale = ops.row_scale(None, Bq, Nq, q.device)
    sums0 = torch.zeros(2, dtype=torch.float64, device="cuda")
    N0 = R.nonneg_fused_chunk(q, v, T, lo, coef, True, sums0)
    clip0, idx0 = ops.maxmean_fwd(q, v, scale, T, want_idx=True)
    clip1, idx1, N1, sums1 = ops.maxmean_fwd_nonneg(q, v, scale, T, lo, coef)
    assert torch.equal(clip0, clip1)
    assert torch.equal(idx0.view(Bv, Bq, -1)[:, :, :Nq], idx1.view(Bv, Bq, -1)[:, :, :Nq])     # (beyond Nq: padding)
    assert torch.equal(N0, N1) and torch.equal(sums0, sums1)
    # gate: nothing flows where the bf16-rounded similarity is below the floor
    S_ref = (raw.bfloat16().float() * 1.5).bfloat16().float()
    assert (N1[S_ref < lo] == 0).all()
    assert (N1[(S_ref < 0) & (S_ref >= lo)] != 0).all()


def test_full_loss_uses_the_merged_forward_and_matches_the_separate_passes():
    """compute_all_similarities_* + compute_contrastive_loss_* with the regularisers on: the merged forward (default)
    and the separate regulariser pass give the same loss and gradients (same kernels' arithmetic, one GEMM each)."""
    import triad_b200
    from triad_b200 import regularizers as R
    from triad_b200.model import TokenSims
    res = {}
    for kind in ("av", "tv"):
        Bq, Nq, Nv, D = (12, 50, 256, 512) if kind == "av" else (10, 77, 256, 512)
        q, v = _inputs(Bq, Bq, Nq, Nv, D, 3)
        mask = None
        if kind == "tv":
            lens = torch.randint(8, Nq + 1, (Bq,), generator=torch.Generator().manual_seed(1))
            mask = (torch.arange(Nq)[None, :] < lens[:, None]).to(torch.int64).cuda()
        for merged in (True, False):
            R.MERGE_FORWARD = merged
            try:
                m = triad_b200.TriadHotPath(1.5, 0.01, 0.5).cuda()
                qd, vd = q.clone().requires_grad_(), v.clone().requires_grad_()
                if kind == "av":
                    clip, tok = m.compute_all_similarities_av(qd, vd)
                    assert (tok.nonneg is not None) == merged
                    total = m.compute_contrastive_loss_av(clip, tok)[0]
                else:
                    clip, tok = m.compute_all_similarities_tv(qd, vd, mask)
                    assert (tok.nonneg is not None) == merged
                    total = m.compute_contrastive_loss_tv(clip, tok)[0]
                assert isinstance(tok, TokenSims) and tok.nonneg is None          # handed over (and freed) by the loss
                total.backward()
                res[(kind, merged)] = (total.item(), qd.grad.float().clone(), vd.grad.float().clone(), m.temperature.grad.item())
            finally:
                R.MERGE_FORWARD = True
        a, b = res[(kind, True)], res[(kind, False)]
        assert abs(a[0] - b[0]) <= 1e-6 * abs(b[0])
        assert ((a[1] - b[1]).norm() / b[1].norm()).item() < 4e-3               # bf16 roundings of the summands differ
        assert ((a[2] - b[2]).norm() / b[2].norm()).item() < 4e-3
        assert abs(a[3] - b[3]) <= 1e-4 * abs(b[3]) + 1e-7


def test_handle_reuse_and_retained_graph():
    """The handle hands N over once: a second loss call on the same handle falls back to the separate regulariser pass
    and gives the same value; backward twice through a retained graph accumulates exactly twice the gradient."""
    import triad_b200
    q, v = _inputs(8, 8, 50, 256, 512, 21)
    m = triad_b200.TriadHotPath(1.5).cuda()
    qd, vd = q.clone().requires_grad_(), v.clone().requires_grad_()
    clip, tok = m.compute_all_similarities_av(qd, vd)
    assert tok.nonneg is not None
    t1 = m.compute_contrastive_loss_av(clip, tok)[0]
    assert tok.nonneg is None
    t2 = m.compute_contrastive_loss_av(clip, tok)[0]
    assert abs(t1.item() - t2.item()) <= 1e-6 * abs(t1.item())
    t1.backward(retain_graph=True)
    g1 = qd.grad.float().clone()
    t1.backward()
    g2 = qd.grad.float()
    assert ((g2 - 2 * g1).norm() / g1.norm()).item() < 8e-3          # bf16 accumulation of two equal gradients
    # evaluation without gradients never takes the merged path (nothing to hand over)
    with torch.no_grad():
        clip3, tok3 = m.compute_all_similarities_av(q, v)
        assert tok3.nonneg is None
        t3 = m.compute_contrastive_loss_av(clip3, tok3)[0]
    assert abs(t3.item() - t1.item()) <= 1e-5 * abs(t1.item())
