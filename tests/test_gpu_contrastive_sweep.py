"""GPU tier: the contrastive step — the max-mean forward (K1), the InfoNCE head (K2), dQ (K3a), dV (K3b) and dT (K3c)
— per element against fp64, on every route its shapes take.  Each step case runs through the drop-in
(``triad_regularizers = False``) or, where a route needs a test flag, through the ``ops.*`` entry points, and asserts
the route it took (``ROUTES``): the kernels it launched, recorded with ``torch.profiler`` in a short run of its own,
and the host rules that no kernel name shows (tile order, dV query blocks and image batches, dT CTAs), restated here.

Rounding model (``tests.helpers.model_sims``): S = bf16(bf16(<q, v>) * T) for bf16 inputs, T * <q, v> for fp32 ones.
u = 2^-24 is the fp32 unit roundoff.  Bounds, per element:

* Winners.  The reference's argmax of S, computed on the device in query chunks from fp64 dot products.  A
  disagreement is allowed only as a certified near-tie (``certify_near_ties``: the two exact dot products are less than
  2 bf16 ulps of the accumulator apart), at most max(2, 1e-4 of the rows); the reference is then pinned to the
  kernel's winners.  Zero-weight rows are not compared (nothing depends on them; a packed forward skips them).
* clip[i, j] = sum_a s_a S[i, j, a, w]: within Nq u sum_a |s_a S| (fp32 summation of <= Nq weighted maxima) plus, for
  each winner whose fp32 accumulator may round to bf16 either way (``ambiguous_bf16_rounding``, or a certified
  near-tie), 2 ulps of S times its weight (one ulp of the accumulator is less than 2 ulps of S after the multiply by
  T).  The window is 32 sigma of a round-to-nearest random walk, 32 * 2^-24 * sqrt(D <q^2, v^2>): the tensor cores
  do not round their fp32 accumulation to nearest (a single S one ulp off outside a 4-sigma window was seen in one
  clip entry of 49 at 7 x 33 x 256 x 512), and 32 sigma also covers a truncation of the running sum after every 16
  products.  fp32 inputs: (D + 2) u T <|q|, |v|> s_a per winner instead (the
  worst case of a D-term fp32 dot product and the multiply by T).
* Head, against fp64 InfoNCE of the kernel's own fp32 clip (so head errors stay apart from forward errors).  A
  log-sum-exp l = m + log(sum_k exp(x_k - m)) over B fp32 terms is within e_l = e_sum + u (2 |l| + 2 log B + 4), with
  e_sum = u (B/32 + rpb + nblk + 8 + sum_k p_k |x_k - m|) the relative error of the sum (sequential and tree adds, the
  rounding of each x_k - m weighted by its softmax share p_k, the exp and log ulps).  Each exp term E = exp(x - l)
  is then within E (e_l + u |x - l| + 3 u), and g = (E_row + E_col - 2 delta) / (2B) within the two terms' bounds
  plus 3 u (E_row + E_col + 2 delta), over 2B, plus 4 fp32 denormal steps where a term underflows.  The loss sum_i (l_row - x_ii) + (l_col - x_ii) / (2B) is within the
  sum of the two l bounds and u |l - x_ii| per term, over 2B, plus u |loss|: where the diagonal dominates this is an
  absolute bound in ulps of |l|.  The fp64 sums of the statistics are within 4 n 2^-53 of their magnitudes; the
  hardest negative is a max of fp32 values and must be bit-equal.
* dq[r, :] = T s_r sum_j g[i, j] v[j, w, :] and dv[j, p, :] = sum_{r: w = p} T s_r g[i, j] q[r, :], from the kernel's
  winners and its g, in fp64: within one bf16 output rounding, 2^-8 of the element (none for fp32 outputs), plus
  (n + 4) u times the same formula on |g|, |v| (|q|), n being the number of terms an fp32 accumulator adds (Bv for dq,
  the (j, p) list length for dv, plus one add per query block where the fp32 scratch collects them).  Padded text
  rows must be exactly zero.
* dT = sum g clip / T: within 1e-5 sum |g clip| / T.
* End to end: where fp64 autograd of the whole step fits (argmax pinned, S rounded as a straight-through offset), the
  drop-in's gradients per block of 128 query rows x 256 columns / one image x 256 columns, within 2^-7 of the
  block's norm for bf16 (1e-5 for fp32), with a floor at 1e-3 of the whole gradient's norm.

Each case prints one JSON line (pytest -s): its routes and how close each check came to its bound.
"""
import json
import math
from dataclasses import dataclass
from typing import Optional

import pytest
import torch

from oracle import oracle as O
from tests import helpers as H
from tests.test_gpu_full_loss_sweep import _blocks_q, _blocks_v, _check_grad

BF, F32 = torch.bfloat16, torch.float32
U = 2.0 ** -24
FWD_SIMT, FWD_1CTA, FWD_SYNC = 1, 2, 8
BWD_SMALL_BLOCKS, BWD_PACK_ROWS = 16, 32
B200_SMS = 148
ACC_WIDTH = 32.0        # ambiguity window of an fp32 tensor-core accumulator, in random-walk sigmas

#: every route of the contrastive step, and what selects it
ROUTES = {
    "fwd:tc_cta2": "tcgen05 forward, cta_group::2",
    "fwd:tc_cta1_size": "tcgen05 forward, cta_group::1 because M = Bq*Nq <= 128",
    "fwd:tc_cta1_flag": "tcgen05 forward, cta_group::1 by TRIAD_FWD_FORCE_1CTA",
    "fwd:simt_fp32": "CUDA-core forward: fp32 inputs",
    "fwd:simt_d%64": "CUDA-core forward: bf16 with D % 64 != 0",
    "fwd:simt_d>512": "CUDA-core forward: bf16 with D > 512",
    "fwd:packed": "masked text: zero-weight rows dropped before the tensor cores",
    "fwd:order_contiguous": "tile order: V <= 48 MB, any order",
    "fwd:order_per_cluster": "tile order: each cluster keeps to its own images",
    "fwd:order_sync": "tile order: chunk-synchronous, selected by size",
    "fwd:order_sync_short": "chunk-synchronous with a short last chunk",
    "fwd:sub_tiles": "Nv > 256: 256-patch sub-tiles with a running max",
    "fwd:nv1": "one patch per image",
    "head:fused": "B <= 2048: triad_contrastive_head",
    "head:blockwise": "B > 2048: infonce_partial / infonce_finish through the drop-in",
    "dq:pipe": "shared-memory pipeline, Nv <= 256",
    "dq:pipe_packed": "shared-memory pipeline over the 8-row groups holding a kept row",
    "dq:tile": "L1-resident gather, Nv > 256",
    "dq:generic_k1": "generic gather, one 32-lane chunk of D",
    "dq:generic_k2": "generic gather, two chunks",
    "dq:generic_k3": "generic gather, three chunks",
    "dq:generic_k4": "generic gather, four chunks",
    "dv:grouped_narrow": "grouped shared-memory sort, D <= 256",
    "dv:grouped_wide": "grouped shared-memory sort, D > 256",
    "dv:many_groups": "more than one 8192-row sort group per query block",
    "dv:global": "global sort (bf16, Nv 1025..3072)",
    "dv:generic": "global sort and the generic gather (fp32)",
    "dv:scratch": "several query blocks summed in an fp32 scratch",
    "dv:image_batches_short": "several image batches, the last one short",
    "dT:one_cta": "dT in one CTA",
    "dT:several_short": "dT in several CTAs, the last chunk short",
    "dT:cap": "dT at its 128-CTA cap (B > 1448)",
}


@dataclass
class Case:
    name: str
    dtype: torch.dtype
    B: int
    Nq: int
    Nv: int
    D: int
    T: float
    mask: Optional[str] = None       # None (audio) | "ragged" | "holes" (zeros inside captions and all-zero captions)
    entry: str = "dropin"            # "dropin" | "ops"
    fwd_flags: int = 0
    bwd_flags: int = 0
    ties: bool = False               # duplicated patches in different 256-patch sub-tiles: exact ties
    seed: int = 0


CASES = [
    Case("cfg2_256x250x256x512", BF, 256, 250, 256, 512, 1.5),
    Case("cfg3_512x77x256x512_masked", BF, 512, 77, 256, 512, 1.5, mask="ragged"),
    Case("av_7x33x256x512", BF, 7, 33, 256, 512, 1.2),
    Case("av_cta1_size_2x64x256x128", BF, 2, 64, 256, 128, 1.5),
    Case("av_cta1_flag_7x33x200x256", BF, 7, 33, 200, 256, 0.9, fwd_flags=FWD_1CTA),
    Case("tv_packed_holes_24x77x256x512", BF, 24, 77, 256, 512, 1.3, mask="holes"),
    Case("tv_packed_nq1_24x1x256x512", BF, 24, 1, 256, 512, 1.1, mask="holes"),
    Case("av_fp32_d128", F32, 7, 33, 64, 128, 0.8),
    Case("tv_fp32_d256_holes", F32, 5, 9, 40, 256, 1.3, mask="holes"),
    Case("av_fp32_d384", F32, 5, 9, 40, 384, 1.1),
    Case("av_fp32_d512_nv300", F32, 5, 9, 300, 512, 1.1),
    Case("av_d72", BF, 24, 33, 64, 72, 1.5),
    Case("av_d264", BF, 5, 9, 40, 264, 1.2),
    Case("av_d520", BF, 5, 9, 40, 520, 1.2),
    Case("tv_d776", BF, 5, 9, 40, 776, 1.2, mask="ragged"),
    Case("tv_d768_holes", BF, 7, 33, 256, 768, 1.2, mask="holes"),
    Case("av_d1024", BF, 5, 20, 128, 1024, 0.8),
    Case("av_nv257_ties", BF, 5, 70, 257, 128, 1.5, ties=True),
    Case("av_nv1024_ties", BF, 5, 70, 1024, 128, 1.5, ties=True),
    Case("av_nv1025_ties", BF, 5, 70, 1025, 128, 1.5, ties=True),
    Case("av_nv3072_ties", BF, 5, 20, 3072, 128, 1.5, ties=True),
    Case("av_nv1", BF, 7, 33, 1, 64, 1.1),
    Case("av_per_cluster_64x64x1024x512", BF, 64, 64, 1024, 512, 1.2, ties=True),
    Case("av_sync_short_200x16x256x512", BF, 200, 16, 256, 512, 1.2),
    Case("av_sync_flag_7x33x256x128", BF, 7, 33, 256, 128, 1.2, fwd_flags=FWD_SYNC),
    Case("av_scratch_300x250x256x512", BF, 300, 250, 256, 512, 1.5),
    Case("av_batches_45x2x2048x1024", BF, 45, 2, 2048, 1024, 1.2, entry="ops", bwd_flags=BWD_SMALL_BLOCKS),
    Case("tv_small_blocks_20x77x200x256", BF, 20, 77, 200, 256, 1.3, mask="ragged", entry="ops",
         bwd_flags=BWD_SMALL_BLOCKS),
    Case("av_blockwise_2049x2x8x64", BF, 2049, 2, 8, 64, 1.1),
    Case("av_blockwise_4096x2x8x64", BF, 4096, 2, 8, 64, 1.3),
]


# ---- host rules, restated ---------------------------------------------------------------------------------------------
def _cdiv(a, b):
    return -(-a // b)


def _align(x, a=256):
    return _cdiv(x, a) * a


def _nq_pad(Nq):
    return _cdiv(Nq, 16) * 16


def _tc_forward(c):
    return c.dtype == BF and not (c.fwd_flags & FWD_SIMT) and c.D % 64 == 0 and 64 <= c.D <= 512


def _packed_forward(c):
    """The drop-in packs masked bf16 text (model.py _similarities); capi.cu packs only on the tensor-core path."""
    return c.entry == "dropin" and c.mask is not None and c.dtype == BF and _tc_forward(c)


def _cta_group(c):
    """capi.cu: a packed forward uses cta_group::2 unless forced; fwd_cta_group: M <= 128 or the flag gives 1."""
    if c.fwd_flags & FWD_1CTA:
        return 1
    return 2 if _packed_forward(c) or c.B * c.Nq > 128 else 1


def _tile_order(c, sms):
    """maxmean_tc.cu pick_tile_order (and the TRIAD_FWD_SYNC_CHUNKS test flag): (order, images per chunk)."""
    if c.fwd_flags & FWD_SYNC:
        return "sync", min(c.B, 3)
    cg = _cta_group(c)
    n_m, n_clusters, img = _cdiv(c.B * c.Nq, 128 * cg), sms // cg, c.Nv * c.D * 2
    if c.B * img <= 48 << 20:
        return "contiguous", c.B
    c16 = max(1, (16 << 20) // img)
    if n_m * c16 >= 4 * n_clusters:
        return "sync", min(c16, c.B)
    return "per_cluster", min(max(1, (48 << 20) // (n_clusters * img)), 64, c.B)


def _dv_plan(Bq, Bv, Nq, Nv, D, elt, out_f32, block_bytes=64 << 20):
    """maxmean_bwd.cu dv_plan: query blocks of <= block_bytes of q, image batches bounding the entry list to 1 GiB
    (and the fp32 scratch to 256 MB)."""
    qb = min(max(1, block_bytes // (Nq * D * elt)), Bq)
    nblk = _cdiv(Bq, qb)
    scratch = nblk > 1 and not out_f32
    ng = _cdiv(qb * _nq_pad(Nq), 8192)
    me = max(ng * 8192, qb * Nq)
    jb = (1 << 30) // (me * 8)
    if scratch:
        jb = min(jb, (256 << 20) // (Nv * D * 4))
    jb = min(max(jb, 1), Bv)
    total = (4096 + 2 * _align(jb * 8 * Nv * 4) + _align(jb * (Nv + 1) * 4) + _align(jb * ng * (Nv + 1) * 4)
             + _align(jb * me * 8) + (_align(jb * Nv * D * 4) if scratch else 0))
    return {"qb": qb, "nblk": nblk, "scratch": scratch, "jb": jb, "groups": ng, "total": total}


def _bwd_workspace_bytes(Bq, Bv, Nq, Nv, D, elt):
    """triad_maxmean_bwd_workspace_bytes: the largest plan over the output types and block sizes, then the packing maps."""
    best = max(_dv_plan(Bq, Bv, Nq, Nv, D, elt, f32, bb)["total"] for f32 in (False, True) for bb in (64 << 20, 64 << 10))
    return best + _align((Bq + 1 + Bq * Nq) * 4 + Bq * 4)


def _case_plan(c):
    small = c.bwd_flags & BWD_SMALL_BLOCKS
    return _dv_plan(c.B, c.B, c.Nq, c.Nv, c.D, c.dtype.itemsize, c.dtype == F32, 64 << 10 if small else 64 << 20)


def _dt_ctas(B):
    """maxmean_bwd.cu: dT_kernel CTAs of 16384 elements, at most 128; (CTAs, elements per CTA, uncapped count)."""
    n = B * B
    nb = min(_cdiv(n, 16384), 128)
    return nb, _cdiv(n, nb), _cdiv(n, 16384)


def _head_rows_per_block(B):
    """infonce.cu head_rows_per_block."""
    rpb = 4
    while _cdiv(B, rpb) > 16:
        rpb *= 2
    while rpb > 32 and _cdiv(B, rpb // 2) <= 64:
        rpb //= 2
    return rpb


def _bwd_pack(c):
    return (c.entry == "dropin" and c.mask is not None and c.dtype == BF) or bool(c.bwd_flags & BWD_PACK_ROWS)


def _predict_routes(c, sms=B200_SMS):
    r = set()
    if not _tc_forward(c):
        r.add("fwd:simt_fp32" if c.dtype == F32 else ("fwd:simt_d%64" if c.D % 64 else "fwd:simt_d>512"))
    else:
        cg = _cta_group(c)
        r.add("fwd:tc_cta2" if cg == 2 else ("fwd:tc_cta1_flag" if c.fwd_flags & FWD_1CTA else "fwd:tc_cta1_size"))
        if _packed_forward(c):
            r.add("fwd:packed")
        order, C = _tile_order(c, sms)
        if order == "sync" and c.fwd_flags & FWD_SYNC:
            order = "sync_flag"
        r.add("fwd:order_" + order)
        if order.startswith("sync") and c.B % C:
            r.add("fwd:order_sync_short")
        if c.Nv > 256:
            r.add("fwd:sub_tiles")
    if c.Nv == 1:
        r.add("fwd:nv1")
    r.add("head:fused" if c.B <= 2048 else "head:blockwise")
    elems = 16 // c.dtype.itemsize
    if c.dtype == BF and c.D % 64 == 0:
        r.add(("dq:pipe_packed" if _bwd_pack(c) else "dq:pipe") if c.Nv <= 256 else "dq:tile")
    else:
        r.add(f"dq:generic_k{_cdiv(c.D // elems, 32)}")
    pl = _case_plan(c)
    if c.dtype == BF:
        if c.Nv <= 1024:
            r.add("dv:grouped_wide" if c.D > 256 else "dv:grouped_narrow")
            if pl["groups"] > 1:
                r.add("dv:many_groups")
        else:
            r.add("dv:global")
    else:
        r.add("dv:generic")
    if pl["scratch"]:
        r.add("dv:scratch")
    if pl["jb"] < c.B and c.B % pl["jb"]:
        r.add("dv:image_batches_short")
    nb, per, uncapped = _dt_ctas(c.B)
    if nb == 1:
        r.add("dT:one_cta")
    elif uncapped > 128:
        r.add("dT:cap")
    elif c.B * c.B % per:
        r.add("dT:several_short")
    return r


def _visible(routes):
    """The part of a route set that kernel names show."""
    out = set()
    for t in routes:
        if t.startswith("fwd:tc_cta1"):
            out.add("fwd:tc_cta1")
        elif t.startswith("fwd:simt"):
            out.add("fwd:simt")
        elif t in ("fwd:tc_cta2", "fwd:packed", "fwd:sub_tiles", "head:fused", "head:blockwise", "dv:global",
                   "dv:generic", "dv:scratch") or t.startswith("dq:"):
            out.add(t)
        elif t.startswith("dv:grouped"):
            out.add("dv:grouped")
    return out


def _routes_from_kernels(names):
    import re
    r = set()
    for n in names:
        m = re.search(r"maxmean_tc_kernel<(\d), (true|false)", n)
        if m:
            r.add("fwd:tc_cta2" if m.group(1) == "2" else "fwd:tc_cta1")
            if m.group(2) == "true":
                r.add("fwd:sub_tiles")
        if "maxmean_simt_kernel" in n:
            r.add("fwd:simt")
        if "pack_copy_kernel" in n:
            r.add("fwd:packed")
        if "nce_head_kernel" in n:
            r.add("head:fused")
        if "nce_finish_kernel" in n:
            r.add("head:blockwise")
        m = re.search(r"dq_gather_kernel<[^<>]*?(\d)>", n)
        if m:
            r.add("dq:generic_k" + m.group(1))
        if "dq_tile_kernel" in n:
            r.add("dq:tile")
        if "dv_group_sort_kernel" in n:
            r.add("dv:grouped")
        if "dv_count_kernel" in n:
            r.add("dv:global")
        if re.search(r"dv_gather_kernel\b", n) or "dv_gather_kernel<" in n:
            r.add("dv:generic")
        if "dv_convert_kernel" in n:
            r.add("dv:scratch")
    if any("dq_pipe_kernel" in n for n in names):
        r.add("dq:pipe_packed" if any("pack_group_map_kernel" in n for n in names) else "dq:pipe")
    if "dv:generic" in r:
        r.discard("dv:global")                 # the generic gather walks the global sort's list
    return r


# ---- inputs and the step --------------------------------------------------------------------------------------------
def _inputs(c):
    g = torch.Generator(device="cuda").manual_seed(2000 + c.seed + 7 * c.B + 11 * c.Nq + 13 * c.Nv + c.D)
    std = math.sqrt(2.0 / (c.T * math.sqrt(c.D)))             # S = T <q, v> with standard deviation ~2
    q = (torch.randn(c.B, c.Nq, c.D, generator=g, device="cuda") * std).to(c.dtype)
    v = (torch.randn(c.B, c.Nv, c.D, generator=g, device="cuda") * std).to(c.dtype)
    if c.ties:                                                 # exact duplicates in different sub-tiles
        v[:, c.Nv - 3] = v[:, 1]
        v[:, 300 % c.Nv] = v[:, 7]
        v[:, c.Nv - 1] = v[:, 2]
    mask = None
    if c.mask is not None:
        lens = torch.randint(1, c.Nq + 1, (c.B,), generator=g, device="cuda")
        lens[0] = c.Nq
        mask = (torch.arange(c.Nq, device="cuda")[None, :] < lens[:, None]).to(torch.int64)
        if c.mask == "holes":
            mask[1, c.Nq // 2: c.Nq // 2 + 2] = 0
            mask[c.B - 1] = 0                                  # an all-zero caption: clamp(sum, 1e-7), a zero clip row
    return q, v, mask


def _head(clip, T):
    """The head the drop-in runs on the kernel's clip: (g, sums fp64 [8], loss).  Deterministic, so for a drop-in case
    this is bit for bit the g its backward used."""
    from triad_b200 import ops
    B = clip.shape[0]
    if B <= ops.HEAD_MAX_B:
        g, sums, out = ops.contrastive_head(clip, None if T is None else torch.tensor(T, device="cuda"))
        return g, sums, out[0].item()
    row_lse, col_part = ops.infonce_partial(clip, B, 0)
    g, sums = ops.infonce_finish(clip, B, 0, row_lse, col_part.reshape(1, 2, B))
    return g, sums, (sums[0] / (2 * B)).to(torch.float32).item()


def _step(c, q, v, mask):
    """One contrastive step: {clip, idx, scale, g, sums, loss, stats, dq, dv, dT}."""
    import triad_b200
    from triad_b200 import ops
    from triad_b200.model import _stats_from_sums
    prefix = "av" if c.mask is None else "tv"
    if c.entry == "dropin":
        m = triad_b200.TriadHotPath(c.T).cuda()
        m.triad_regularizers = False
        m.triad_fwd_flags = c.fwd_flags
        qd, vd = q.clone().requires_grad_(), v.clone().requires_grad_()
        if c.mask is None:
            clip_out, tok = m.compute_all_similarities_av(qd, vd)
            res = m.compute_contrastive_loss_av(clip_out, tok)
            con, stats = res[1], res[4]
        else:
            clip_out, tok = m.compute_all_similarities_tv(qd, vd, mask)
            con, stats = m.compute_contrastive_loss_tv(clip_out, tok)
        con.backward()
        clip = tok.clip.detach()
        g, sums, loss = _head(clip, c.T if c.mask is None else None)
        assert con.item() == loss
        return {"clip": clip, "idx": tok.idx_t, "scale": tok.row_scale, "g": g, "sums": sums, "loss": loss,
                "stats": dict(stats), "dq": qd.grad, "dv": vd.grad, "dT": m.temperature.grad.item()}
    scale = ops.row_scale(mask, c.B, c.Nq, q.device)
    Tt = torch.tensor(c.T, device="cuda")
    clip, idx = ops.maxmean_fwd(q, v, scale, Tt, flags=c.fwd_flags)
    g, sums, loss = _head(clip, c.T if c.mask is None else None)
    dq, dv, dT = ops.maxmean_bwd(q, v, idx, g, clip, scale, Tt, flags=c.bwd_flags)
    return {"clip": clip, "idx": idx, "scale": scale, "g": g, "sums": sums, "loss": loss,
            "stats": _stats_from_sums(sums, c.B, prefix), "dq": dq, "dv": dv, "dT": dT.item()}


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}


# ---- checks ---------------------------------------------------------------------------------------------------------
def _assert_within(err, bound, what, worst):
    ratio = (err / bound.clamp(min=1e-300)).nan_to_num(nan=float("inf"))
    worst[what] = max(worst.get(what, 0.0), ratio.max().item() if ratio.numel() else 0.0)
    bad = (err > bound) | err.isnan()
    if bool(bad.any()):
        k = bad.nonzero()[0].tolist()
        raise AssertionError(f"{what}: {int(bad.sum())} elements out of bound, first at {k}: "
                             f"err {err[tuple(k)].item():.3e} > bound {bound[tuple(k)].item():.3e}")


def _check_forward(c, q, v, scale64, got_w, clip, worst):
    """Winners and clip per element; returns the winners the backward reference uses (the kernel's, certified)."""
    B, Nq, Nv, D = c.B, c.Nq, c.Nv, c.D
    live = scale64 > 0
    v64 = v.double()
    ci = max(1, (1 << 25) // (B * Nq * Nv))
    n_bad, gap = 0, 0.0
    for i0 in range(0, B, ci):
        i1 = min(B, i0 + ci)
        qc = q[i0:i1].double()
        raw = torch.einsum("iad,jpd->ijap", qc, v64)
        S = H.model_sims(raw, c.T, c.dtype)
        ref_w = S.argmax(dim=3)
        got = torch.where(live[i0:i1, None, :], got_w[i0:i1], ref_w)
        nb, wg = H.certify_near_ties(q[i0:i1], v, got, ref_w)
        n_bad, gap = n_bad + nb, max(gap, wg)
        got_w[i0:i1] = got
        pick = lambda t: t.gather(3, got[..., None]).squeeze(3)
        Sw, rw = pick(S), pick(raw)
        w = scale64[i0:i1, None, :]
        if c.dtype == BF:
            sq = pick(torch.einsum("iad,jpd->ijap", qc * qc, v64 * v64))
            amb = H.ambiguous_bf16_rounding(rw, sq, D, width=ACC_WIDTH) | (got != ref_w)
            slack = (torch.where(amb, 2 * H.bf16_ulp(Sw), torch.zeros_like(Sw)) * w).sum(2)
        else:
            ab = pick(torch.einsum("iad,jpd->ijap", qc.abs(), v64.abs()))
            slack = ((D + 2) * U * c.T * ab * w).sum(2)
        ref = (Sw * w).sum(2)
        bound = Nq * U * (Sw.abs() * w).sum(2) + slack
        _assert_within((clip[i0:i1].double() - ref).abs(), bound, "clip", worst)
    assert n_bad <= max(2, 1e-4 * B * B * Nq), n_bad
    assert gap < 2.0, gap
    worst["argmax flips"] = n_bad
    return got_w


def _lse_bound(x, lse, dim, B, rpb, nblk):
    """Bound on the fp32 log-sum-exp of x along dim (see the module docstring)."""
    m = x.max(dim=dim, keepdim=True).values
    p = torch.exp(x - lse)
    e_sum = U * (B / 32 + rpb + nblk + 8 + (p * (x - m).abs()).sum(dim=dim, keepdim=True))
    return e_sum + U * (2 * lse.abs() + 2 * math.log(B) + 4)


def _check_head(clip, g, sums, loss, stats, prefix, worst, rpb=32, nblk=None):
    """g, the loss, the fp64 sums and the six statistics of the head on the fp32 clip, against fp64."""
    x = clip.double()
    B = x.shape[0]
    nblk = _cdiv(B, rpb) if nblk is None else nblk
    lse_r, lse_c = torch.logsumexp(x, 1, keepdim=True), torch.logsumexp(x, 0, keepdim=True)
    er, ec = torch.exp(x - lse_r), torch.exp(x - lse_c)
    eye = torch.eye(B, dtype=torch.float64, device=x.device)
    g64 = (er + ec - 2 * eye) / (2 * B)
    b_r, b_c = _lse_bound(x, lse_r, 1, B, rpb, nblk), _lse_bound(x, lse_c, 0, B, rpb, nblk)
    e_er = er * (b_r + U * (x - lse_r).abs() + 3 * U)
    e_ec = ec * (b_c + U * (x - lse_c).abs() + 3 * U)
    bound_g = (e_er + e_ec + 3 * U * (er + ec + 2 * eye)) / (2 * B) + 4 * 2.0 ** -149   # exp terms below fp32's range
    _assert_within((g.double() - g64).abs(), bound_g, "g", worst)
    d = torch.diagonal(x)
    lr, lc = lse_r.reshape(-1), lse_c.reshape(-1)
    loss64 = ((lr - d).sum() + (lc - d).sum()) / (2 * B)
    per = torch.diagonal(b_r.expand(B, B)) + torch.diagonal(b_c.expand(B, B)) + U * ((lr - d).abs() + (lc - d).abs())
    bound_sum = per.sum()
    _assert_within((sums[0] - 2 * B * loss64).abs().reshape(1), (bound_sum + 1e-300).reshape(1), "loss sum", worst)
    bound_loss = bound_sum / (2 * B) + U * loss64.abs()
    _assert_within(torch.tensor([abs(loss - loss64.item())]), (bound_loss + 1e-300).reshape(1).cpu(), "loss", worst)
    off = x[~torch.eye(B, dtype=torch.bool, device=x.device)]
    tiny = 4 * B * B * 2.0 ** -53
    want = torch.stack([d.sum(), (d * d).sum(), off.sum(), (off * off).sum()])
    mag = torch.stack([d.abs().sum(), (d * d).sum(), off.abs().sum(), (off * off).sum()])
    _assert_within((sums[1:5] - want).abs(), tiny * mag + 1e-300, "stat sums", worst)
    gc_bound = (bound_g * x.abs()).sum() + tiny * (g64 * x).abs().sum()
    _assert_within((sums[6] - (g64 * x).sum()).abs().reshape(1), (gc_bound + 1e-300).reshape(1), "sum g*clip", worst)
    if off.numel():                                           # B = 1: see test_single_pair_batch_statistics
        hardest, want_h = sums[5].item(), off.max().item()
        assert hardest == want_h or (math.isnan(hardest) and math.isnan(want_h)), (hardest, want_h)
    ref = O.similarity_stats(x.cpu(), prefix)
    assert sorted(stats) == sorted(ref)
    n_d, n_o = B, off.numel()
    bounds = {"pos_sim_mean": tiny * d.abs().mean().item(), "neg_sim_mean": tiny * off.abs().mean().item() if n_o else 0,
              "pos_sim_std": tiny * (d * d).mean().item() * n_d / max(n_d - 1, 1),
              "neg_sim_std": tiny * (off * off).mean().item() * n_o / max(n_o - 1, 1) if n_o else 0}
    bounds["separation"] = bounds["pos_sim_mean"] + bounds["neg_sim_mean"]
    for k, want_k in ref.items():
        key = k[len(prefix) + 1:]
        got_k = stats[k]
        if math.isnan(want_k):
            assert math.isnan(got_k), (k, got_k)
            continue
        if key == "hardest_negative":
            assert got_k == want_k, (k, got_k, want_k)
        elif key.endswith("std"):                              # compare variances: the std of a constant is 0
            e = abs(got_k * got_k - want_k * want_k)
            assert e <= bounds[key] + 1e-300, (k, got_k, want_k)
        else:
            assert abs(got_k - want_k) <= bounds[key] + 1e-300, (k, got_k, want_k)
    return bound_g, bound_loss.item()


def _check_backward(c, q, v, scale64, winners, out, plan, worst):
    B, Nq, Nv, D, T = c.B, c.Nq, c.Nv, c.D, c.T
    R = 2.0 ** -8 if c.dtype == BF else 0.0                  # one bf16 rounding of the output (unit roundoff)
    g64 = out["g"].double()
    q64, vflat = q.double(), v.double().reshape(B * Nv, D)
    dq = out["dq"].double().reshape(B, Nq, D)
    base = (torch.arange(B, device="cuda") * Nv)[None, :, None]
    dv_ref = torch.zeros(B * Nv, D, dtype=torch.float64, device="cuda")
    dv_mag, cnt = torch.zeros_like(dv_ref), torch.zeros(B * Nv, dtype=torch.float64, device="cuda")
    ci = max(1, (1 << 25) // (B * Nq * D))
    for i0 in range(0, B, ci):
        i1 = min(B, i0 + ci)
        flat = winners[i0:i1] + base                                                    # (ci, Bv, Nq)
        w = T * scale64[i0:i1, None, :] * g64[i0:i1, :, None]
        vg = vflat[flat]
        ref = (w[..., None] * vg).sum(1)
        mag = (w.abs()[..., None] * vg.abs()).sum(1)
        del vg
        _assert_within((dq[i0:i1] - ref).abs(), R * ref.abs() + (1 + R) * (B + 4) * U * mag, "dq", worst)
        qe = q64[i0:i1, None].expand(-1, B, -1, -1)
        fl = flat.reshape(-1)
        dv_ref.index_add_(0, fl, (w[..., None] * qe).reshape(-1, D))
        dv_mag.index_add_(0, fl, (w.abs()[..., None] * qe.abs()).reshape(-1, D))
        cnt.index_add_(0, fl, (scale64[i0:i1, None, :] > 0).expand_as(w).reshape(-1).double())
    if c.mask is not None:                                    # padded tokens: exactly zero gradient
        assert bool((out["dq"][(scale64 == 0)] == 0).all())
    n = cnt[:, None] + plan["nblk"] + 4
    dv = out["dv"].double().reshape(B * Nv, D)
    _assert_within((dv - dv_ref).abs(), R * dv_ref.abs() + (1 + R) * n * U * dv_mag, "dv", worst)
    gc = g64 * out["clip"].double()
    _assert_within(torch.tensor([abs(out["dT"] - gc.sum().item() / T)]),
                   torch.tensor([1e-5 * gc.abs().sum().item() / T + 1e-300]), "dT", worst)


def _check_end_to_end(c, q, v, scale64, winners, out, worst):
    """fp64 autograd of the whole contrastive step with the argmax pinned, per gradient block."""
    B, Nq, Nv, D = c.B, c.Nq, c.Nv, c.D
    q64, v64 = q.double().requires_grad_(), v.double().requires_grad_()
    flat = winners + (torch.arange(B, device="cuda") * Nv)[None, :, None]
    raw = (q64[:, None] * v64.reshape(B * Nv, D)[flat]).sum(-1)
    S = raw * c.T
    if c.dtype == BF:
        S = S + (H.model_sims(raw.detach(), c.T, c.dtype) - S).detach()
    clip = (S * scale64[:, None, :]).sum(-1)
    d = torch.diagonal(clip)
    loss = ((torch.logsumexp(clip, 1) - d).sum() + (torch.logsumexp(clip, 0) - d).sum()) / (2 * B)
    gq, gv = torch.autograd.grad(loss, [q64, v64])
    tol = 2.0 ** -7 if c.dtype == BF else 1e-5
    _check_grad(out["dq"], gq.reshape(B * Nq, D), _blocks_q(c), tol, "e2e dq", worst, 1e-300)
    _check_grad(out["dv"], gv.reshape(B * Nv, D), _blocks_v(c), tol, "e2e dv", worst, 1e-300)


E2E_MAX = 6e7           # B*B*Nq*D of the fp64 autograd graph (about 0.5 GB per tensor)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_contrastive_step_against_fp64(case):
    from triad_b200 import ops
    c = case
    torch.cuda.reset_peak_memory_stats()
    q, v, mask = _inputs(c)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    routes = _predict_routes(c, sms)
    seen = _routes_from_kernels(_kernel_names(lambda: _step(c, q, v, mask)))
    assert seen == _visible(routes), (sorted(seen), sorted(_visible(routes)))
    out = _step(c, q, v, mask)
    # the kernels' row weights are the reference's (model.py:509-512 in fp32)
    if mask is None:
        want_scale = torch.full((c.B, c.Nq), 1.0 / c.Nq, device="cuda")
    else:
        m = mask.float()
        want_scale = m / m.sum(dim=1, keepdim=True).clamp(min=1e-7)
    assert torch.equal(out["scale"].view(c.B, c.Nq), want_scale)
    scale64 = want_scale.double()
    worst = {}
    winners = _check_forward(c, q, v, scale64, ops.idx_to_reference_layout(out["idx"], c.B, c.Nq), out["clip"], worst)
    rpb = _head_rows_per_block(c.B) if c.B <= 2048 else 32
    _check_head(out["clip"], out["g"], out["sums"], out["loss"], out["stats"], "av" if mask is None else "tv", worst,
                rpb=rpb)
    _check_backward(c, q, v, scale64, winners, out, _case_plan(c), worst)
    if c.entry == "dropin" and c.B * c.B * c.Nq * c.D <= E2E_MAX:
        _check_end_to_end(c, q, v, scale64, winners, out, worst)
    print(json.dumps({"case": c.name, "routes": sorted(routes), "worst_over_bound": worst,
                      "peak_mem_gb": round(torch.cuda.max_memory_allocated() / 1e9, 2)}))


def test_every_route_is_covered():
    """Every row of ROUTES is taken by at least one case (each case asserts its routes against the kernels it ran)."""
    seen = {}
    for c in CASES:
        for r in _predict_routes(c):
            seen.setdefault(r, []).append(c.name)
    missing = sorted(set(ROUTES) - set(seen))
    assert not missing, missing
    assert set(seen) - {"fwd:order_sync_flag"} <= set(ROUTES), set(seen) - set(ROUTES)
    # cfg 2 takes the chunk-synchronous order by size (V = 67 MB), not by the test flag
    assert "fwd:order_sync" in _predict_routes(CASES[0]) and CASES[0].fwd_flags == 0
    for B in (1, 2, 15, 16, 17, 33, 255, 256, 257, 1025, 2047, 2048):
        assert B in HEAD_BS
    assert {B for B in BLOCKWISE_BS if B > 2048} and any(1 in cuts for _, cuts in SHARD_CUTS)


@pytest.mark.parametrize("shape", [(256, 256, 250, 256, 512), (512, 512, 77, 256, 512), (300, 300, 250, 256, 512),
                                   (45, 45, 2, 2048, 1024), (20, 20, 77, 200, 256), (4096, 4096, 2, 8, 64),
                                   (1100, 4, 250, 32, 64), (7, 7, 33, 64, 128), (5, 5, 9, 300, 512)])
@pytest.mark.parametrize("dtype", [1, 0])
def test_dv_plan_restatement_matches_the_library(shape, dtype):
    """The restated dv_plan (query blocks, image batches, fp32 scratch) gives the library's workspace size, byte for
    byte, so the routes the step cases claim from it are the ones the library takes."""
    from triad_b200 import _lib, build
    build.build()
    lib = _lib.load()
    Bq, Bv, Nq, Nv, D = shape
    elt = 2 if dtype == 1 else 4
    assert lib.triad_maxmean_bwd_workspace_bytes(Bq, Bv, Nq, Nv, D, dtype) == _bwd_workspace_bytes(Bq, Bv, Nq, Nv, D, elt)


def test_single_pair_batch_statistics():
    """B = 1 has no off-diagonal entry: the negative statistics and the hardest negative are NaN (the reference's max
    over an empty tensor raises; the oracle returns NaN)."""
    from triad_b200.model import _stats_from_sums
    x = 0.75
    sums = torch.tensor([0.0, x, x * x, 0.0, 0.0, float("-inf"), 0.0, 0.0], dtype=torch.float64)
    got = _stats_from_sums(sums, 1, "av")
    want = O.similarity_stats(torch.tensor([[x]]), "av")
    for k, w in want.items():
        assert (math.isnan(w) and math.isnan(got[k])) or got[k] == w, (k, got[k], w)
    assert math.isnan(got["av_hardest_negative"])


# ---- the InfoNCE head on its own ------------------------------------------------------------------------------------
HEAD_BS = [1, 2, 15, 16, 17, 33, 255, 256, 257, 1025, 2047, 2048]
BLOCKWISE_BS = [2049, 4096, 8192]
KINDS = ["n0.01", "n2", "n30", "diag50", "const", "bf16"]
SHARD_CUTS = [(64, [32, 32]), (100, [1, 50, 49]), (257, [40, 1, 30, 30, 50, 6, 60, 40]), (4100, [4000, 99, 1]),
              (2048, [256] * 8)]


def _synthetic_clip(B, kind, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed + B)
    if kind == "const":
        return torch.full((B, B), 0.3, device="cuda")
    sigma = {"n0.01": 0.01, "n2": 2.0, "n30": 30.0, "diag50": 1.0, "bf16": 2.0}[kind]
    x = torch.randn(B, B, generator=g, device="cuda") * sigma
    if kind == "diag50":
        x += 50 * torch.eye(B, device="cuda")
    if kind == "bf16":                                        # an edited AV clip: bf16 values, honoured as given
        x = x.bfloat16().float()
    return x


def _poisoned(shape):
    """Leave a NaN-filled block of this size at the top of the caching allocator, so that an output the kernel
    forgets to write reads NaN rather than a previous call's values."""
    t = torch.full(shape, float("nan"), device="cuda")
    del t


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("B", HEAD_BS)
def test_fused_head_against_fp64(B, kind):
    from triad_b200 import ops
    from triad_b200.model import _stats_from_sums
    clip = _synthetic_clip(B, kind)
    _poisoned((B, B))
    g, sums, out = ops.contrastive_head(clip, None)
    worst = {}
    rpb = _head_rows_per_block(B)
    _check_head(clip, g, sums, out[0].item(), _stats_from_sums(sums, B, "av"), "av", worst, rpb=rpb,
                nblk=_cdiv(B, rpb))
    if kind == "const":                                       # loss log B, g = (2/B - 2 delta) / (2B)
        assert abs(out[0].item() - math.log(B)) <= 8 * U * max(math.log(B), 1) + 1e-7
    print(json.dumps({"head": "fused", "B": B, "kind": kind, "worst_over_bound": worst}))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["n2", "n30", "diag50", "const"])
@pytest.mark.parametrize("B", BLOCKWISE_BS)
def test_blockwise_head_against_fp64(B, kind):
    from triad_b200 import ops
    from triad_b200.model import _stats_from_sums
    clip = _synthetic_clip(B, kind)
    row_lse, col_part = ops.infonce_partial(clip, B, 0)
    _poisoned((B, B))
    g, sums = ops.infonce_finish(clip, B, 0, row_lse, col_part.reshape(1, 2, B))
    worst = {}
    _check_head(clip, g, sums, (sums[0] / (2 * B)).float().item(), _stats_from_sums(sums, B, "tv"), "tv", worst)
    print(json.dumps({"head": "blockwise", "B": B, "kind": kind, "worst_over_bound": worst}))


def _sharded_head(clip, cuts):
    """dist.sharded_contrastive_step's head on one GPU: a row block per rank with its row0, the column partials of all
    blocks stacked, then each block's finish.  Returns (g, all_sums [W, 8])."""
    from triad_b200 import ops
    B = clip.shape[0]
    r0s = [sum(cuts[:k]) for k in range(len(cuts))]
    parts = [ops.infonce_partial(clip[r0:r0 + n].contiguous(), B, r0) for r0, n in zip(r0s, cuts)]
    col_parts = torch.stack([p[1] for p in parts])
    gs, sums = [], []
    for (r0, n), (row_lse, _) in zip(zip(r0s, cuts), parts):
        _poisoned((n, B))
        g, s = ops.infonce_finish(clip[r0:r0 + n].contiguous(), B, r0, row_lse, col_parts)
        gs.append(g)
        sums.append(s)
    return torch.cat(gs), torch.stack(sums)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["n2", "diag50", "bf16"])
@pytest.mark.parametrize("B,cuts", SHARD_CUTS, ids=[f"B{B}-W{len(c)}" for B, c in SHARD_CUTS])
def test_row_sharded_head_against_fp64(B, cuts, kind):
    from triad_b200 import dist, ops
    assert sum(cuts) == B
    clip = _synthetic_clip(B, kind, seed=len(cuts))
    g, all_sums = _sharded_head(clip, cuts)
    loss = (all_sums[:, 0].sum() / (2 * B)).to(torch.float32).item()
    worst = {}
    sums = dist.combine_all_sums(all_sums)
    bound_g, bound_loss = _check_head(clip, g, sums, loss, dist.stats_from_all_sums(all_sums, B, "av"), "av", worst,
                                      nblk=_cdiv(B, 32) + len(cuts))
    # and the unsharded call: the same to fp32 rounding (each is within its bound of fp64)
    row_lse, col_part = ops.infonce_partial(clip, B, 0)
    g1, s1 = ops.infonce_finish(clip, B, 0, row_lse, col_part.reshape(1, 2, B))
    assert bool(((g.double() - g1.double()).abs() <= 2 * bound_g).all())
    assert abs(loss - (s1[0] / (2 * B)).to(torch.float32).item()) <= 2 * bound_loss
    assert s1[5].item() == sums[5].item()
    print(json.dumps({"head": "sharded", "B": B, "W": len(cuts), "kind": kind, "worst_over_bound": worst}))


@pytest.mark.gpu
@pytest.mark.parametrize("route", ["fused", "blockwise", "sharded"])
def test_nan_clip_entry_reaches_loss_g_and_hardest_negative(route):
    """One NaN off the diagonal: the loss, that row and that column of g are NaN — and so is the hardest negative, as
    the reference's torch max gives it; every other g entry stays finite."""
    from triad_b200 import dist, ops
    from triad_b200.model import _stats_from_sums
    B = 33 if route == "fused" else 2049
    clip = _synthetic_clip(B, "n2")
    i, j = 3, 7
    clip[i, j] = float("nan")
    if route == "fused":
        g, sums, out = ops.contrastive_head(clip, None)
        loss = out[0].item()
        stats = _stats_from_sums(sums, B, "av")
    elif route == "blockwise":
        row_lse, col_part = ops.infonce_partial(clip, B, 0)
        g, sums = ops.infonce_finish(clip, B, 0, row_lse, col_part.reshape(1, 2, B))
        loss = (sums[0] / (2 * B)).item()
        stats = _stats_from_sums(sums, B, "av")
    else:
        g, all_sums = _sharded_head(clip, [1000, 1049])
        loss = (all_sums[:, 0].sum() / (2 * B)).item()
        stats = dist.stats_from_all_sums(all_sums, B, "av")
    assert math.isnan(loss)
    assert bool(g[i].isnan().all()) and bool(g[:, j].isnan().all())
    rest = torch.ones(B, B, dtype=torch.bool, device="cuda")
    rest[i] = False
    rest[:, j] = False
    assert bool(g[rest].isfinite().all())
    assert math.isnan(O.similarity_stats(clip.cpu(), "av")["av_hardest_negative"])
    assert math.isnan(stats["av_hardest_negative"])


@pytest.mark.gpu
def test_single_pair_batch_head():
    """B = 1: loss 0, g 0, and the statistics of test_single_pair_batch_statistics from the kernel's sums."""
    from triad_b200 import ops
    from triad_b200.model import _stats_from_sums
    clip = torch.tensor([[0.75]], device="cuda")
    g, sums, out = ops.contrastive_head(clip, None)
    assert out[0].item() == 0.0 and g.item() == 0.0
    stats = _stats_from_sums(sums, 1, "av")
    assert stats["av_pos_sim_mean"] == 0.75 and math.isnan(stats["av_hardest_negative"])
    assert math.isnan(stats["av_neg_sim_mean"]) and math.isnan(stats["av_separation"])
