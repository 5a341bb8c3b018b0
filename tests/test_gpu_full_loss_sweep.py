"""GPU tier: the reference's FULL training loss — symmetric InfoNCE of the max-mean similarities plus the
regularisers (dense non-negative pressure, temporal smoothness / patch-usage sparsity on the positive pairs, the
temperature-calibration term) — through the two public entry points, the drop-in loss methods and
``dist.sharded_full_loss_step`` at world size 1, against an fp64 autograd evaluation of the same loss.

The cases are organised by the route the dense regulariser takes (see ``ROUTES``); each case records the route it
actually took, read from the handle (``TokenSims.nonneg``) and from which kernels ran, and
``test_every_route_is_covered`` asserts that every route has a case.

Reference.  fp64 autograd on the device: S = T * <q, v> for every token pair, the oracle's ``regularization_av`` /
``regularization_tv`` on S, and InfoNCE of the max-mean similarity with the argmax pinned to the winners the GPU chose
(each disagreement with the reference's own argmax first certified as a near-tie: the two candidates' exact dot
products are less than 2 bf16 ulps apart).  For bf16 inputs S is rounded like the reference under autocast,
S = bf16(bf16(<q, v>) * T), as a straight-through offset S64 + (round(S64) - S64).detach(): values and the clamp gate
follow the rounded S, gradients stay exact.

Bounds, from the rounding model:

* fp32 inputs: every value within 1e-5 relative; gradients within 1e-5 relative per block (below).
* bf16 inputs: the product sees the same rounded S as the reference except where an fp32 accumulator sits within its
  own error of a bf16 rounding boundary (rare; one S moves by one ulp, 2^-8 relative), and evaluates the terms in
  fp32 / fp64 from there.  Values: within 2^-13 (1.2e-4) relative, plus, for every S whose first rounding an fp32
  accumulator may take either way (<q, v> within 4 sigma of the accumulator's random-walk rounding error,
  2^-22 * sqrt(D * <q^2, v^2>), of a bf16 rounding midpoint), one ulp of S times |d value / dS| (a few such S decide
  a mean over a handful of elements at the smallest shapes).  Away from the clamp floor the tcgen05 dense-term
  forward evaluates S = T * acc in fp32 rather than rounding it twice (maxmean_tc.cu): an unbiased difference of at
  most 2^-8 |S| per pair, so the dense term's value also gets 4 sigma of that random walk,
  4 * 2^-8 * ||dl_nonneg/dS * S||_2 (at the 2 x 2 x 8 shape this is what decides the bound).
  Gradients: the product returns them in bf16 (one rounding, <= 2^-9 relative per element), built from bf16
  intermediates (N = dL/d<q,v> of the dense term and G of the positive-pair term, <= 2^-9 each) and, in the
  drop-in, summed in bf16 by autograd (<= 2^-9 of each part): within 2^-7 (7.8e-3) relative per block.
* Gradient blocks: the query gradient in blocks of 128 token rows x 256 columns, the image gradient per image x 256
  columns.  A block's error is bounded relative to that block's reference norm, with a floor at 1e-3 of the whole
  gradient's norm, so one wrong tile, image chunk or column half fails on its own.
* dT of each term: within the same relative bound of that term's magnitude sum_{S} |dterm/dS * S| / T (+ |dl_cal/dT|):
  dT is a sum over every token pair that can cancel.

Every case proves its terms are non-trivial in the reference: negative similarities for the dense term, some patch
usage fraction above the threshold for the sparsity term (the threshold and weight are chosen per case from the
reference's fractions), smoothness > 0.
"""
import math
import random
from dataclasses import dataclass, field
from typing import Tuple

import pytest
import torch

from oracle import oracle as O
from tests import helpers as H

pytestmark = pytest.mark.gpu

#: every route the full loss can take, and what selects it
ROUTES = {
    "merged": "drop-in: one pass for max-mean and the dense term (triad_maxmean_fwd_nonneg), own GEMMs",
    "fused_chunked": "drop-in: separate tcgen05 dense forward (triad_nonneg_fused_chunk) over several image chunks, "
                     "fp32 dQ accumulator (N over the chunk budget)",
    "fused_zpad": "drop-in: the separate tcgen05 dense forward on images padded with zero patches (Nv % 8 != 0)",
    "mm_own_gemm": "drop-in: library GEMM + triad_nonneg_chunk, own backward GEMMs (Nv > 256 or D % 64 != 0, D <= 512)",
    "mm_torch_gemm": "drop-in: library GEMM + triad_nonneg_chunk + library backward GEMMs (D > 512)",
    "fp32": "drop-in: fp32 inputs",
    "sharded_merged": "sharded_full_loss_step: merged pass, one image chunk",
    "sharded_merged_chunked": "sharded_full_loss_step: merged pass, several image chunks, the last one short",
    "sharded_composed": "sharded_full_loss_step: sharded_contrastive_step + sharded_regularizer_step",
}

BF16_VALUE_TOL, BF16_GRAD_TOL = 2.0 ** -13, 2.0 ** -7
FP32_VALUE_TOL, FP32_GRAD_TOL = 1e-5, 1e-5
Q_BLOCK_ROWS, COL_BLOCK = 128, 256


@dataclass
class Case:
    name: str
    kind: str                    # "av" | "tv"
    dtype: torch.dtype
    B: int
    Nq: int
    Nv: int
    D: int
    T: float
    amp: float = 2.0             # standard deviation of S = T <q, v>
    mask: str = "none"           # tv: "ragged" | "holes" (zeros inside captions and one all-zero caption)
    small_chunks: bool = False   # drop-in: a chunk budget below the batch's N (several image chunks)
    sharded: Tuple[str, ...] = ("one",)     # "one" | "several" | "composed"
    seed: int = 0
    info: dict = field(default_factory=dict)


BF, F32 = torch.bfloat16, torch.float32
FIXED = [
    Case("av_merged_7x33x256x512", "av", BF, 7, 33, 256, 512, 0.8, sharded=("one", "several", "composed")),
    Case("tv_merged_24x77x256x512", "tv", BF, 24, 77, 256, 512, 1.3, mask="ragged", sharded=("one", "several", "composed")),
    Case("av_merged_nv8_24x250x8x64", "av", BF, 24, 250, 8, 64, 1.5, sharded=("one", "several")),
    Case("av_merged_b1", "av", BF, 1, 250, 256, 512, 0.9),
    Case("av_merged_b2_nq2", "av", BF, 2, 2, 8, 64, 1.2, sharded=("one", "several")),
    Case("tv_merged_nq1", "tv", BF, 24, 1, 256, 512, 0.7, mask="ragged", sharded=("one", "several")),
    Case("tv_zpad_holes_24x77x201x128", "tv", BF, 24, 77, 201, 128, 1.2, mask="holes"),
    Case("av_zpad_7x250x201x192", "av", BF, 7, 250, 201, 192, 0.7),
    Case("av_zpad_tiny_2x2x13x64", "av", BF, 2, 2, 13, 64, 1.5),
    Case("tv_zpad_nv1", "tv", BF, 7, 33, 1, 64, 1.1, mask="ragged"),
    Case("av_zpad_chunked_7x33x201x512", "av", BF, 7, 33, 201, 512, 0.9, small_chunks=True),
    Case("av_fused_chunked_7x77x256x512", "av", BF, 7, 77, 256, 512, 0.9, small_chunks=True),
    Case("tv_fused_chunked_d320", "tv", BF, 7, 33, 200, 320, 1.4, mask="holes", small_chunks=True),
    Case("av_mm_nv257", "av", BF, 7, 33, 257, 512, 0.8),
    Case("tv_mm_nv600_d264", "tv", BF, 7, 77, 600, 264, 1.3, mask="ragged"),
    Case("av_mm_d72", "av", BF, 24, 33, 64, 72, 1.5),
    Case("av_d768", "av", BF, 7, 33, 128, 768, 0.8),
    Case("tv_d768", "tv", BF, 7, 33, 256, 768, 1.2, mask="holes"),
    Case("av_fp32", "av", F32, 7, 33, 64, 128, 0.8),
    Case("tv_fp32_holes", "tv", F32, 7, 77, 201, 64, 1.3, mask="holes"),
    Case("av_clamp_floor", "av", BF, 7, 33, 64, 128, 1.5, amp=40.0, sharded=("one", "several")),
    Case("tv_clamp_floor", "tv", BF, 7, 33, 64, 128, 1.5, amp=15.0, mask="ragged", sharded=("one", "several")),
]


def _random_cases(n, seed=20261021):
    rng = random.Random(seed)
    out = []
    while len(out) < n:
        kind = rng.choice(["av", "tv"])
        B, Nq = rng.choice([1, 2, 7, 24]), rng.choice([1, 2, 33, 77, 250])
        Nv, D = rng.choice([1, 8, 13, 201, 256, 257, 600]), rng.choice([64, 72, 192, 264, 320, 512, 768])
        dtype = BF if rng.random() < 0.8 else F32
        if B * B * Nq * Nv > 3e7 or (kind == "av" and Nq == 1):      # av with one token: see test_single_token_av
            continue
        if dtype == F32 and D > 512:                                 # the fp32 backward takes D <= 512 (loud error)
            continue
        T = rng.choice([0.6, 0.9, 1.2, 1.7])
        mask = rng.choice(["ragged", "holes"]) if kind == "tv" else "none"
        out.append(Case(f"rand{len(out)}_{kind}_{'bf16' if dtype == BF else 'fp32'}_{B}x{Nq}x{Nv}x{D}", kind, dtype,
                        B, Nq, Nv, D, T, amp=rng.choice([1.0, 2.0, 4.0]), mask=mask,
                        small_chunks=rng.random() < 0.3 and B > 1, sharded=("one", "several") if B > 1 else ("one",),
                        seed=len(out) + 100))
    return out


CASES = FIXED + _random_cases(8)
RUNS = [(c, entry) for c in CASES for entry in ("dropin",) + tuple("sharded_" + s for s in c.sharded)]


# ---- inputs ---------------------------------------------------------------------------------------------------------
def _inputs(c: Case):
    g = torch.Generator(device="cuda").manual_seed(1000 + c.seed + 7 * c.B + 11 * c.Nq + 13 * c.Nv + c.D)
    std = math.sqrt(c.amp / (c.T * math.sqrt(c.D)))          # S = T <q, v> has standard deviation amp
    q = (torch.randn(c.B, c.Nq, c.D, generator=g, device="cuda") * std).to(c.dtype)
    v = (torch.randn(c.B, c.Nv, c.D, generator=g, device="cuda") * std).to(c.dtype)
    mask = None
    if c.kind == "tv":
        lens = torch.randint(1, c.Nq + 1, (c.B,), generator=g, device="cuda")
        lens[0] = c.Nq
        mask = (torch.arange(c.Nq, device="cuda")[None, :] < lens[:, None]).to(torch.int64)
        if c.mask == "holes":
            mask[0, c.Nq // 2: c.Nq // 2 + 2] = 0
            if c.B > 2:
                mask[c.B - 1] = 0                           # an all-zero caption: clamp(sum, 1e-7), a zero clip row
    return q, v, mask


def _row_scale64(c, mask):
    if mask is None:
        return torch.full((c.B, c.Nq), 1.0 / c.Nq, dtype=torch.float64, device="cuda")
    m = mask.to(torch.float32)
    return (m / m.sum(dim=1, keepdim=True).clamp(min=1e-7)).double()        # model.py:509-512 in fp32


def _rounded_sims(q, v, T):
    """(raw fp64 <q,v>, S with the product's rounding as a straight-through offset, T64 leaf, q64, v64 leaves)."""
    q64 = q.detach().double().requires_grad_()
    v64 = v.detach().double().requires_grad_()
    T64 = torch.tensor(float(T), dtype=torch.float64, device="cuda", requires_grad=True)
    raw = torch.einsum("iad,jpd->ijap", q64, v64)
    S = raw * T64
    if q.dtype == torch.bfloat16:
        Sr = H.model_sims(raw.detach(), T, q.dtype)
        S = S + (Sr - S).detach()
    return raw, S, T64, q64, v64


def _rounding_slack_weights(q, v, raw):
    """Per element: 2 ulps of S where the bf16 rounding of <q, v> is ambiguous under fp32 accumulation, else 0."""
    if q.dtype != torch.bfloat16:
        return None
    with torch.no_grad():
        sq = torch.einsum("iad,jpd->ijap", q.double() ** 2, v.double() ** 2)
        ulp = H.bf16_ulp(raw.float().bfloat16().double())
        ambiguous = H.ambiguous_bf16_rounding(raw, sq, q.shape[-1])
        return torch.where(ambiguous, 2 * ulp, torch.zeros_like(ulp))


def _certified_winners(c, q, v, S, got, scale):
    """The GPU's winners where they are certified near-ties of the reference's own argmax; the reference's argmax on
    zero-weight rows (nothing depends on them; a packed forward leaves them unwritten)."""
    ref = S.detach().argmax(dim=3)
    live = (scale > 0)[:, None, :].expand_as(ref)
    got = torch.where(live, got.clamp(0, c.Nv - 1), ref)
    n_bad, worst = H.certify_near_ties(q, v, got, ref)
    assert n_bad <= max(2, 1e-4 * ref.numel()), n_bad
    assert worst < 2.0, worst
    return got


def _threshold_and_weight(c, S, mask):
    """tv: a threshold between the smallest and the largest patch usage fraction (so relu(frac - thr) is neither
    all zero nor everywhere active) and a weight that gives the sparsity term the dense term's size."""
    with torch.no_grad():
        diag = S[torch.arange(c.B), torch.arange(c.B)]
        frac = torch.softmax(diag, dim=-1).sum(dim=1) / c.Nq
        thr = min(float(frac.flatten().quantile(0.75)), 0.9 * float(frac.max()))
        excess = torch.relu(frac - thr).pow(2).mean().item()
        nonneg = S.clamp(min=-20, max=0).pow(2).mean().item()
        w = 0.15 * nonneg / excess if excess > 0 else 1.0
    return thr, min(max(w, 1e-3), 1e6)


def _reference(c, q, v, mask, thr, w, winners, drop_single_row_smooth=False):
    raw, S, T64, q64, v64 = _rounded_sims(q, v, c.T)
    amb = _rounding_slack_weights(q, v, raw.detach())
    scale = _row_scale64(c, mask)
    best = S.gather(3, winners[..., None]).squeeze(3)                       # (B, B, Nq)
    clip = (best * scale[:, None, :]).sum(dim=2)
    lse_r, lse_c, d = torch.logsumexp(clip, 1), torch.logsumexp(clip, 0), torch.diagonal(clip)
    con = ((lse_r - d).sum() + (lse_c - d).sum()) / (2 * c.B)
    lo = -60.0 if c.kind == "av" else -20.0
    nonneg = 0.15 * S.clamp(min=lo, max=0).pow(2).mean()
    diag = S[torch.arange(c.B), torch.arange(c.B)]
    if c.kind == "av":
        cal = 20 * torch.clamp(-torch.log(T64), min=0) ** 2
        if c.Nq > 1 or not drop_single_row_smooth:
            reg, pos = O.regularization_av(S, T64)                          # pos = 0.01 * l_smooth
        else:
            reg, pos = cal + nonneg, torch.zeros((), dtype=torch.float64, device="cuda")
        frac = None
    else:
        cal = torch.zeros((), dtype=torch.float64, device="cuda")
        reg = O.regularization_tv(S, thr, w)
        frac = torch.softmax(diag.detach(), dim=-1).sum(dim=1) / c.Nq
        pos = w * torch.relu(torch.softmax(diag, dim=-1).sum(dim=1) / c.Nq - thr).pow(2).mean()
    if not math.isnan(reg.item()):
        assert abs(reg.item() - (cal + nonneg + pos).item()) <= 1e-12 * abs(reg.item())
    total = con + reg
    terms = {"total": total, "contrastive": con, "reg": reg, "pos": pos, "nonneg": nonneg}
    out = {k: t.item() for k, t in terms.items()}
    T = float(c.T)
    dcal = torch.autograd.grad(cal, T64, retain_graph=True)[0].item() if cal.requires_grad else 0.0
    mag = {"cal": abs(dcal)}                  # sum over S of |d term / dS * S| / T: what dT of the term sums up
    for name in ("contrastive", "nonneg", "pos"):
        t = terms[name]
        gS = torch.autograd.grad(t, S, retain_graph=True)[0] if t.requires_grad and math.isfinite(t.item()) else None
        mag[name] = 0.0 if gS is None else (gS.abs() * S.detach().abs()).sum().item() / T
        out["slack_" + name] = 0.0 if (gS is None or amb is None) else (gS.abs() * amb).sum().item() * T
        if name == "nonneg" and amb is not None and gS is not None:   # fp32 S in the tcgen05 dense emission
            out["slack_nonneg"] += 4 * 2.0 ** -8 * (gS * S.detach()).norm().item()
    mag["reg"] = mag["cal"] + mag["nonneg"] + mag["pos"]
    out["slack_reg"] = out["slack_nonneg"] + out["slack_pos"]
    out["slack_total"] = out["slack_contrastive"] + out["slack_reg"]
    mag["total"] = mag["contrastive"] + mag["reg"]
    grads = {}
    for name in ("total", "reg", "contrastive", "pos"):
        t = terms[name]
        if not t.requires_grad or not math.isfinite(t.item()):
            continue
        gq, gv, gT = torch.autograd.grad(t, [q64, v64, T64], retain_graph=True, allow_unused=True)
        zero = lambda x, like: torch.zeros_like(like) if x is None else x
        grads[name] = {"dq": zero(gq, q64), "dv": zero(gv, v64), "dT": 0.0 if gT is None else gT.item(),
                       "dT_mag": mag[name]}
    # anti-vacuity: every term of this case carries weight
    out["neg_frac"] = (S.detach() < 0).double().mean().item()
    out["below_floor"] = (S.detach() < lo).double().mean().item()
    out["frac_max"] = None if frac is None else frac.max().item()
    out["frac_over"] = None if frac is None else (frac > thr).double().mean().item()
    return out, grads


# ---- the two entry points -------------------------------------------------------------------------------------------
class _Counter:
    def __init__(self):
        self.n = {}

    def wrap(self, mp, obj, name):
        fn = getattr(obj, name)

        def counted(*a, **k):
            self.n[name] = self.n.get(name, 0) + 1
            return fn(*a, **k)
        mp.setattr(obj, name, counted)


def _run_dropin(c, q, v, mask, thr, w, monkeypatch, want_grads=True):
    import triad_b200
    from triad_b200 import ops
    from triad_b200 import regularizers as R
    cnt = _Counter()
    for obj, name in ((R, "nonneg_fused_chunk"), (R, "nonneg_chunk"), (ops, "dense_grad_gemm")):
        cnt.wrap(monkeypatch, obj, name)
    if c.small_chunks:             # room for about half the images' N: several chunks, the last one short
        nv_pad = (c.Nv + 7) // 8 * 8
        jc = max(1, (c.B - 1) // 2)
        monkeypatch.setattr(R, "CHUNK_BYTES", jc * c.B * c.Nq * nv_pad * q.element_size())
    m = triad_b200.TriadHotPath(c.T, thr, w).cuda()
    m.triad_regularizers = True

    def forward():
        qd, vd = q.clone().requires_grad_(), v.clone().requires_grad_()
        if c.kind == "av":
            clip, tok = m.compute_all_similarities_av(qd, vd)
        else:
            clip, tok = m.compute_all_similarities_tv(qd, vd, mask)
        return qd, vd, clip, tok

    # the loss call a training step makes
    qd, vd, clip, tok = forward()
    merged = tok.nonneg is not None
    if c.kind == "av":
        total, con, reg, smooth, _ = m.compute_contrastive_loss_av(clip, tok)
        vals = {"total": total.item(), "contrastive": con.item(), "reg": reg.item(), "pos": smooth.item()}
    else:
        total, _ = m.compute_contrastive_loss_tv(clip, tok)
        vals = {"total": total.item()}
    n_fused, n_mm, n_gemm = (cnt.n.get(k, 0) for k in ("nonneg_fused_chunk", "nonneg_chunk", "dense_grad_gemm"))
    if merged:
        route = "merged"
    elif n_fused:
        route = "fused_zpad" if c.Nv % 8 else "fused_chunked"
    elif q.dtype == torch.float32:
        route = "fp32"
    else:
        route = "mm_own_gemm" if n_gemm else "mm_torch_gemm"
    c.info.update(route=route, chunks=max(n_fused, n_mm, 1))
    if route == "fused_chunked":
        assert n_fused > 1
    if not want_grads:
        return route, None, None, None
    winners = tok.argmax()
    grads = {}
    m.temperature.grad = None
    total.backward()
    grads["total"] = {"dq": qd.grad, "dv": vd.grad, "dT": m.temperature.grad.item()}
    # the regularisers alone and the contrastive part alone, from a second forward
    qd, vd, clip, tok = forward()
    con = m._loss_head(clip, tok, c.kind, False)[0]
    if c.kind == "av":
        reg, smooth = m.compute_regularization_losses_av(tok)
    else:
        reg, smooth = m.compute_regularization_losses_tv(tok), None
    vals.setdefault("contrastive", con.item())
    vals.setdefault("reg", reg.item())
    for name, t in (("reg", reg), ("contrastive", con), ("pos", smooth)):
        if t is None:
            continue
        gq, gv, gT = torch.autograd.grad(t, [qd, vd, m.temperature], retain_graph=True, allow_unused=True)
        grads[name] = {"dq": gq, "dv": gv, "dT": 0.0 if gT is None else gT.item()}
    return route, vals, grads, winners


def _sharded_kernels(force_composed):
    from triad_b200.dist import CudaKernels

    class Recording(CudaKernels):
        """The product kernels; records the chunk count and the argmax buffer, optionally refuses the merged pass."""
        n_chunks = 0
        idx = None

        def full_loss_merged(self, q, v):
            return False if force_composed else super().full_loss_merged(q, v)

        def maxmean_fwd_nonneg(self, *a):
            self.n_chunks += 1
            return super().maxmean_fwd_nonneg(*a)

        def maxmean_fwd(self, q, v, scale, T):
            clip, idx = super().maxmean_fwd(q, v, scale, T)
            self.idx = idx
            return clip, idx

        def maxmean_bwd_dq(self, q, v, idx, g, scale, T):
            self.idx = idx
            return super().maxmean_bwd_dq(q, v, idx, g, scale, T)
    return Recording()


def _run_sharded(c, variant, q, v, mask, thr, w):
    from triad_b200 import ops
    from triad_b200.dist import sharded_full_loss_step
    k = _sharded_kernels(variant == "composed")
    chunk_bytes = None
    if variant == "several":
        jc = max(1, (c.B - 1) // 2)                           # B = 7: 3 + 3 + 1
        chunk_bytes = jc * c.B * c.Nq * c.Nv * 2
    out = sharded_full_loss_step(q, v, torch.tensor(c.T, device="cuda"), c.kind, mask, kernels=k,
                                 patch_sparsity_threshold=thr, patch_sparsity_weight=w, chunk_bytes=chunk_bytes)
    if k.n_chunks == 0:
        route = "sharded_composed"
    else:
        route = "sharded_merged_chunked" if k.n_chunks > 1 else "sharded_merged"
        if variant == "several":
            assert k.n_chunks > 1
    winners = ops.idx_to_reference_layout(k.idx, c.B, c.Nq)
    vals = {"total": out["total"].item(), "contrastive": out["contrastive"].item(), "reg": out["reg"].item()}
    if c.kind == "av":
        vals["pos"] = out["smooth"].item()
    grads = {"total": {"dq": out["dq"], "dv": out["dv"], "dT": out["dT"].item()}}
    assert out["dT_global"].item() == out["dT"].item()       # one rank: its share is all of it
    return route, vals, grads, winners


# ---- comparison -----------------------------------------------------------------------------------------------------
def _blocks_q(c):
    for r0 in range(0, c.B * c.Nq, Q_BLOCK_ROWS):
        for c0 in range(0, c.D, COL_BLOCK):
            yield f"q rows {r0}+ cols {c0}+", (slice(r0, r0 + Q_BLOCK_ROWS), slice(c0, c0 + COL_BLOCK))


def _blocks_v(c):
    for j in range(c.B):
        for c0 in range(0, c.D, COL_BLOCK):
            yield f"image {j} cols {c0}+", (slice(j * c.Nv, (j + 1) * c.Nv), slice(c0, c0 + COL_BLOCK))


def _check_grad(got, ref, blocks, tol, what, worst, abs_floor):
    """Norm-wise, then block by block (relative to the block's reference norm, floor 1e-3 of the whole norm).
    abs_floor: a norm below which the reference counts as zero (B = 1: the contrastive gradient vanishes)."""
    ref = ref.detach().double()
    got = got.detach().double().reshape(ref.shape)
    gnorm = max(ref.norm().item(), abs_floor)
    err = (got - ref).norm().item()
    worst[what] = max(worst.get(what, 0.0), err / (tol * gnorm))
    assert err <= tol * gnorm, (what, err / gnorm)
    floor = 1e-3 * gnorm
    for name, (rs, cs) in blocks:
        e = (got[rs, cs] - ref[rs, cs]).norm().item()
        bound = tol * max(ref[rs, cs].norm().item(), floor)
        worst[what + " block"] = max(worst.get(what + " block", 0.0), e / bound)
        assert e <= bound, (what, name, e, bound)


def _report(case, entry, payload):
    """One JSON line on stdout (shown with pytest -s): the route, the error-to-bound ratio of every check (how close
    each bound sits) and the peak device memory."""
    import json
    print(json.dumps({"case": case.name, "entry": entry, **payload}))


def _compare(c, vals, grads, ref, rgrads):
    fp32 = c.dtype == torch.float32
    vtol, gtol = (FP32_VALUE_TOL, FP32_GRAD_TOL) if fp32 else (BF16_VALUE_TOL, BF16_GRAD_TOL)
    worst = {}
    # values: each relative to the total's magnitude floor of 1e-6 (B = 1: the contrastive part is exactly 0)
    floor = 1e-6 * (abs(ref["contrastive"]) + abs(ref["reg"]))
    for key, got in vals.items():
        want = ref[key]
        bound = vtol * max(abs(want), floor) + ref["slack_" + key]
        worst["value " + key] = abs(got - want) / bound
        assert abs(got - want) <= bound, (key, got, want, ref["slack_" + key])
    tot = rgrads["total"]
    for name, g in grads.items():
        r = rgrads[name]
        if g.get("dq") is not None:
            _check_grad(g["dq"], r["dq"].reshape(c.B * c.Nq, c.D), _blocks_q(c), gtol, f"d{name}/dq", worst,
                        1e-6 * tot["dq"].norm().item())
        if g.get("dv") is not None:
            _check_grad(g["dv"], r["dv"].reshape(c.B * c.Nv, c.D), _blocks_v(c), gtol, f"d{name}/dv", worst,
                        1e-6 * tot["dv"].norm().item())
        bound = gtol * max(r["dT_mag"], 1e-6 * tot["dT_mag"])
        worst[f"d{name}/dT"] = abs(g["dT"] - r["dT"]) / bound
        assert abs(g["dT"] - r["dT"]) <= bound, (name, g["dT"], r["dT"], r["dT_mag"])
    return worst


def _anti_vacuity(c, ref):
    assert ref["neg_frac"] > 0 and ref["nonneg"] > 0            # the dense term sees negative similarities
    if c.kind == "tv":
        assert ref["frac_over"] > 0 and ref["pos"] > 0          # some patch is used more than the threshold
    elif c.Nq > 1:
        assert ref["pos"] > 0                                   # smoothness
    if c.name.endswith("clamp_floor"):
        assert ref["below_floor"] > 1e-3                        # S reaches the clamp floor


@pytest.mark.parametrize("case,entry", RUNS, ids=[f"{c.name}-{e}" for c, e in RUNS])
def test_full_loss_against_fp64(case, entry, monkeypatch):
    c = case
    q, v, mask = _inputs(c)
    raw, S, _, _, _ = _rounded_sims(q, v, c.T)
    thr, w = _threshold_and_weight(c, S.detach(), mask) if c.kind == "tv" else (0.3, 0.1)
    del raw, S
    if entry == "dropin":
        route, vals, grads, got_idx = _run_dropin(c, q, v, mask, thr, w, monkeypatch)
    else:
        route, vals, grads, got_idx = _run_sharded(c, entry[len("sharded_"):], q, v, mask, thr, w)
    raw, S, _, _, _ = _rounded_sims(q, v, c.T)
    winners = _certified_winners(c, q, v, S.detach(), got_idx, _row_scale64(c, mask))
    del raw, S
    ref, rgrads = _reference(c, q, v, mask, thr, w, winners)
    _anti_vacuity(c, ref)
    worst = _compare(c, vals, grads, ref, rgrads)
    _report(c, entry, {"route": route, "worst_over_bound": max(worst.values()), "worst": worst,
                       "peak_mem_gb": torch.cuda.max_memory_allocated() / 1e9})


def test_every_route_is_covered(monkeypatch):
    """Each route of ROUTES is taken by at least one case, as observed while the product runs."""
    seen = {}
    for c in CASES:
        q, v, mask = _inputs(c)
        with monkeypatch.context() as mp:
            route = _run_dropin(c, q, v, mask, 0.5, 0.1, mp, want_grads=False)[0]
        seen.setdefault(route, []).append(c.name)
        for variant in c.sharded:
            route = _run_sharded(c, variant, q, v, mask, 0.5, 0.1)[0]
            seen.setdefault(route, []).append(f"{c.name}/{variant}")
    missing = sorted(set(ROUTES) - set(seen))
    assert not missing, (missing, {k: len(x) for k, x in seen.items()})
    assert set(seen) <= set(ROUTES), set(seen) - set(ROUTES)


def test_single_token_av():
    """Audio with one token has no temporal differences.  The drop-in follows the reference: the smoothness term is
    the mean over an empty tensor, NaN, and so are the regulariser and the total.  sharded_full_loss_step drops the
    term (documented there) and returns the loss without it, which must match fp64."""
    c = Case("av_nq1", "av", BF, 7, 1, 256, 512, 0.8)
    q, v, _ = _inputs(c)
    import triad_b200
    m = triad_b200.TriadHotPath(c.T).cuda()
    clip, tok = m.compute_all_similarities_av(q.clone().requires_grad_(), v.clone().requires_grad_())
    total, con, reg, smooth, _ = m.compute_contrastive_loss_av(clip, tok)
    assert math.isnan(smooth.item()) and math.isnan(reg.item()) and math.isnan(total.item())
    assert math.isfinite(con.item())
    raw, S, T64, _, _ = _rounded_sims(q, v, c.T)
    assert math.isnan(O.regularization_av(S, T64)[1].item())          # the reference's own value
    for variant in ("one", "several"):
        route, vals, grads, got_idx = _run_sharded(c, variant, q, v, None, 0.3, 0.1)
        assert vals["pos"] == 0.0
        winners = _certified_winners(c, q, v, S.detach(), got_idx, _row_scale64(c, None))
        ref, rgrads = _reference(c, q, v, None, 0.3, 0.1, winners, drop_single_row_smooth=True)
        rgrads = {"total": rgrads["total"]}
        _compare(c, vals, grads, ref, rgrads)
