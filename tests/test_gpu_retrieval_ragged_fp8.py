"""GPU tier: retrieval over an e4m3 ragged caption gallery (``RaggedGallery(fp8=True)``, ``triad_ragged_pack_e4m3``,
``triad_retrieve_scores_ragged_e4m3``).

Contract.  Slot row r stores codes c_r and scale s_r from the per-row quantizer (s = fp32(amax / 448), codes
e4m3_rn_satfinite(fp32(x / s))), read in the input's own dtype (fp32 is not rounded to bf16 first); the rows after a
slot's last caption have s = 0 and zero codes.  The query is quantized per token (codes cq, scales sq_a), and acc is
the tensor-core dot product of the codes.
    direction 0 (aggregator_tv_v2t): score_c = sum_a fp32(m_ac t_a),  m_ac = max_{t in c} fp32(s_t acc_at),
        t_a = fp32(fp32(sq_a fp32(1/Nq)) fp32(1/T)), the sum over a in the dense forward's 32-row-group order;
    direction 1 (aggregator_tv_t2v): score_c = sum_{t in c, token order} fp32(m_t w_t),  m_t = max_a fp32(sq_a acc_ta),
        w_t = fp32(fp32(s_t fp32(1/len_c)) fp32(1/T)).
Both maxima propagate NaN: a caption row holding an inf or a NaN makes that caption's score NaN and no other's; a
non-finite query token makes every score NaN.

A. Pack: with fp32 and bf16 input, every caption row's codes and scale are bit-equal to triad_quantize_e4m3 of that
   row; gap rows have zero codes and scale 0; from_padded keeps the masked rows; cat of partly full slots.
B. Exact probe, both directions: small-integer codes, power-of-two scales, Nq, T and caption lengths, so every
   product, weight and fp32 sum is exact and the scores must equal fp64 bit for bit.
C. Per-caption scores against fp64 of the dequantized operands, with the tolerance of tests/test_gpu_retrieval_fp8.py
   for a 24-bit accumulator restated:
       tol_c = (1 + 2^-6) (D 2^-23 B_c + (K + 8) 2^-23 A_c),
   A_c = the score's mean of max |e| (e = the dequantized similarity / T) and B_c the same mean of max
   sq_a s_t sum_k |cq_ak c_tk| / T, K = the number of terms of the mean (Nq in direction 0, the caption's length in
   direction 1).  Shapes: Nq in {1, 77, 129, 256, 1024}, cfg 3's lengths U[8, 77] and galleries of 1-token and
   256-token captions, T in {1.5, 0.07}, slot counts on both sides of the tile-order thresholds (an e4m3 slot is
   256 D bytes, so 48 MB is 384 slots at D = 512).  Each case asserts its kernel path; one test asserts every path
   is reached.
D. Direction 0 equals (==) the Fp8Gallery score of each caption alone, from the same input rows.
E. NaN isolation (a non-finite caption row, a non-finite query token); repeated calls are bit-identical; a caption
   scores the same after another prefix; no host synchronisation; no gallery-sized temporary.
F. Agreement with the bf16 RaggedGallery on a planted gallery, both directions: the planted ids and their order agree
   and the premise gap covers the quantization error.
G. Gallery-sharded top-k: one rank against retrieve_topk; two ranks under NCCL (skipped on one GPU).
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from triad_b200 import _lib, ops, retrieval as R
from triad_b200._lib import check

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = torch.device("cuda")
_SMS = torch.cuda.get_device_properties(0).multi_processor_count if torch.cuda.is_available() else 148
_MiB = 1 << 20
SLOT = 256


def _captions(lengths, D, seed, dtype=torch.bfloat16):
    g = torch.Generator(device=DEV).manual_seed(seed)
    flat = torch.nn.functional.normalize(torch.randn(int(np.sum(lengths)), D, generator=g, device=DEV), dim=1)
    return list(torch.split(flat.to(dtype), [int(x) for x in lengths]))


def _lengths(spec, n, seed):
    if spec == "cfg3":
        return np.random.default_rng(seed).integers(8, 78, size=n)
    return np.full(n, int(spec))


def _quant(x):
    codes = torch.empty(x.shape, dtype=torch.uint8, device=x.device)
    scales = torch.empty(x.shape[:-1], dtype=torch.float32, device=x.device)
    R._quantize_rows(x, codes, scales)
    return codes, scales


def _segments(gal):
    """Caption id of every slot row (n_cap for the zero rows at a slot's end)."""
    info = gal.cap_info.cpu().numpy()
    cid = np.full(gal.n_slots * SLOT, len(gal), dtype=np.int64)
    for c, (r, n) in enumerate(info):
        cid[r:r + n] = c
    return torch.from_numpy(cid).to(DEV)


def _raw(qc, qs, gal, T, direction):
    """triad_retrieve_scores_ragged_e4m3 on given query codes and scales."""
    lib = _lib.load()
    Nq, D = qc.shape
    n_cap = len(gal)
    Tt = ops.temperature_tensor(T, DEV)
    out = torch.empty(n_cap, dtype=torch.float32, device=DEV)
    nws = lib.triad_retrieve_ragged_workspace_bytes(Nq, gal.n_slots, n_cap, direction)
    ws = torch.empty(nws, dtype=torch.uint8, device=DEV)
    check(lib.triad_retrieve_scores_ragged_e4m3(qc.data_ptr(), qs.data_ptr(), Nq, gal.slots.data_ptr(),
                                                gal.scales.data_ptr(), gal.meta.data_ptr(), gal.cap_info.data_ptr(),
                                                gal.n_slots, n_cap, D, Tt.data_ptr(), direction, out.data_ptr(),
                                                ws.data_ptr(), nws, ops._stream(DEV)), "triad_retrieve_scores_ragged_e4m3")
    return out


def _fp64(qc, qs, gal, T):
    """{direction: (score, A, B, K)} per caption in fp64, the operands dequantized exactly."""
    n = len(gal)
    cid = _segments(gal)
    keep = cid < n
    cid = cid[keep]
    c8 = gal.slots.view(torch.uint8)[keep].view(torch.float8_e4m3fn)
    rows = c8.double() * gal.scales[keep].double()[:, None]
    q = qc.view(torch.float8_e4m3fn).double() * qs.double()[:, None]
    e = rows @ q.T / T                                                     # [caption rows, Nq]
    mag = (c8.double().abs() @ qc.view(torch.float8_e4m3fn).double().abs().T)
    mag *= gal.scales[keep].double()[:, None] * qs.double()[None, :] / T
    lens = torch.from_numpy(gal.lengths.astype(np.int64)).to(DEV)

    def segmax(x):
        out = torch.full((n, x.shape[1]), -float("inf"), dtype=torch.float64, device=DEV)
        return out.scatter_reduce_(0, cid[:, None].expand_as(x), x, "amax", include_self=True)

    def segmean(x):
        return torch.zeros(n, dtype=torch.float64, device=DEV).index_add_(0, cid, x) / lens

    Nq = qc.shape[0]
    out = {0: (segmax(e).mean(1), segmax(e.abs()).mean(1), segmax(mag).mean(1),
               torch.full((n,), Nq, dtype=torch.float64, device=DEV))}
    out[1] = (segmean(e.amax(1)), segmean(e.abs().amax(1)), segmean(mag.amax(1)), lens.double())
    return out


def _tolerance(D, A, B, K):
    return (1 + 2.0 ** -6) * (D * 2.0 ** -23 * B + (K + 8) * 2.0 ** -23 * A)


# ----------------------------------------------------------------------------------------------------------------
# which forward path a call takes (launch_maxmean_tc's tile order for e4m3 slots, restated)
# ----------------------------------------------------------------------------------------------------------------
def _path(Nq, n_slots, D, direction, sms=_SMS):
    if direction == 1:                                           # rows = slot rows: cta_group::2, one image
        return "tc2", "default", 1, Nq > 256
    cta = 1 if Nq <= 128 else 2
    n_m = -(-Nq // (128 * cta))
    img = SLOT * D                                               # one byte per e4m3 code
    clusters = sms // cta
    order, C = "default", n_slots
    if n_slots * img > 48 * _MiB:
        c16 = max(1, 16 * _MiB // img)
        if n_m * c16 >= 4 * clusters:
            order, C = "sync", min(c16, n_slots)
        else:
            order, C = "retrieval", min(max(1, min(64, 48 * _MiB // (clusters * img))), n_slots)
    return f"tc{cta}", order, C, False


def _label(kern, order, C, sub):
    return kern + "-" + order + (("-C1" if C == 1 else "-C>1") if order == "retrieval" else "") + ("-sub" if sub else "")


# (Nq, D, lengths, captions, path the direction-0 call is written for).  An e4m3 slot of D = 512 is 128 KB, so no
# one-query shape reaches a one-slot retrieval chunk (C = 1): that needs slots of more than 48 MB / (2 * 148).
_CASES = [
    (77, 512, "cfg3", 600, "tc1-default"),             # ~110 slots, 14 MB: below the 48 MB threshold
    (77, 512, "cfg3", 3000, "tc1-retrieval-C>1"),      # ~550 slots, 70 MB
    (1, 128, "cfg3", 10000, "tc1-retrieval-C>1"),      # one query token, ~1850 slots of 32 KB
    (129, 256, "1", 12800, "tc2-default"),             # 1-token captions: 256 per slot, 50 slots
    (256, 512, "256", 500, "tc2-retrieval-C>1"),       # 256-token captions: one per slot, 64 MB
    (1024, 256, "cfg3", 5000, "tc2-sync"),             # ~920 slots of 64 KB with four query tiles
    (1024, 512, "cfg3", 800, "tc2-default"),           # direction 1: four 256-token sub-tiles of the query
]
_TEMPS = (1.5, 0.07)
_GAL = {}


def _case(ci):
    if ci not in _GAL:
        _GAL.clear()
        torch.cuda.empty_cache()
        Nq, D, spec, n, _ = _CASES[ci]
        gal = R.RaggedGallery.from_list(_captions(_lengths(spec, n, 100 + ci), D, 200 + ci), fp8=True)
        g = torch.Generator(device=DEV).manual_seed(300 + ci)
        q = torch.nn.functional.normalize(torch.randn(Nq, D, generator=g, device=DEV), dim=1).bfloat16()
        qc, qs = _quant(q)
        _GAL[ci] = (q, gal, {T: _fp64(qc, qs, gal, T) for T in _TEMPS})
    return _GAL[ci]


@pytest.fixture(scope="module", autouse=True)
def _release():
    yield
    _GAL.clear()
    torch.cuda.empty_cache()


def test_cases_reach_every_path():
    seen = set()
    for ci, (Nq, D, spec, n, want) in enumerate(_CASES):
        n_slots = R.ragged_plan(_lengths(spec, n, 100 + ci))[0].shape[0]
        assert _label(*_path(Nq, n_slots, D, 0)) == want, (ci, _path(Nq, n_slots, D, 0))
        seen.add(want)
        seen.add(_label(*_path(Nq, n_slots, D, 1)))
    assert {"tc1-default", "tc2-default", "tc1-retrieval-C>1", "tc2-retrieval-C>1", "tc2-sync",
            "tc2-default-sub"} <= seen, seen
    assert {c[0] for c in _CASES} >= {1, 77, 129, 256, 1024}


# ----------------------------------------------------------------------------------------------------------------
# A. pack
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_pack_is_the_row_quantizer(dtype):
    D = 256
    lens = np.array([77, 1, 30, 200, 8, 256, 3, 64] * 3)
    caps = _captions(lens, D, 5, dtype)
    caps[3] = caps[3] * 1000.0                                      # one caption far from unit norm
    gal = R.RaggedGallery.from_list(caps, fp8=True)
    assert gal.slots.dtype == torch.float8_e4m3fn and gal.scales.shape == (gal.n_slots * SLOT,)
    c_ref, s_ref = _quant(torch.cat(caps))                          # fp32 quantized as fp32, not rounded to bf16
    cid = _segments(gal)
    keep = cid < len(gal)
    assert torch.equal(gal.slots.view(torch.uint8)[keep], c_ref)
    assert torch.equal(gal.scales[keep].view(torch.int32), s_ref.view(torch.int32))
    assert (gal.slots.view(torch.uint8)[~keep] == 0).all() and (gal.scales[~keep] == 0).all()
    assert (~keep).any()
    if dtype == torch.float32:                                      # premise: fp32 and its bf16 rounding differ
        cb, _ = _quant(torch.cat(caps).bfloat16())
        assert not torch.equal(cb, c_ref)


def test_from_padded_and_cat_of_partly_full_slots():
    D = 128
    g = torch.Generator(device=DEV).manual_seed(41)
    feats = torch.randn(5, 77, D, generator=g, device=DEV)
    mask = torch.zeros(5, 77, dtype=torch.int64)
    for i, n in enumerate([77, 1, 30, 8, 64]):
        mask[i, :n] = 1
    gal = R.RaggedGallery.from_padded(feats, mask, fp8=True)
    ref = R.RaggedGallery.from_list([feats[i][mask[i].bool().to(DEV)] for i in range(5)], fp8=True)
    assert torch.equal(gal.slots.view(torch.uint8), ref.slots.view(torch.uint8))
    assert torch.equal(gal.scales, ref.scales) and torch.equal(gal.cap_info, ref.cap_info)
    a = R.RaggedGallery.from_list(_captions([100, 50], D, 1), fp8=True)           # one partly full slot
    b = R.RaggedGallery.from_list(_captions([200, 70, 9], D, 2), fp8=True)        # two, the last partly full
    j = R.RaggedGallery.cat([a, b])
    assert torch.equal(j.slots.view(torch.uint8), torch.cat([a.slots, b.slots]).view(torch.uint8))
    assert torch.equal(j.scales, torch.cat([a.scales, b.scales]))
    assert j.n_slots == 3 and len(j) == 5 and j.nbytes == a.nbytes + b.nbytes
    q = torch.randn(40, D, generator=g, device=DEV)
    for d in (0, 1):
        assert torch.equal(R._scores_ragged(q, j, 0.5, d), torch.cat([R._scores_ragged(q, a, 0.5, d),
                                                                       R._scores_ragged(q, b, 0.5, d)]))


# ----------------------------------------------------------------------------------------------------------------
# B. exact probe
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("Nq,D,T", [(4, 128, 0.5), (512, 256, 2.0)])
def test_exact_probe_both_directions(Nq, D, T):
    g = torch.Generator(device=DEV).manual_seed(Nq + D)
    pattern = [1, 2, 64, 4, 128, 32, 8, 16, 256, 1, 1, 32, 64, 128, 2, 4, 8, 16, 32, 1, 256, 2]
    lens = np.array(pattern * 3)
    gal = R.RaggedGallery.from_list(_captions(lens, D, 11), fp8=True)
    keep = _segments(gal) < len(gal)
    rows = int(keep.sum())
    # small-integer codes and power-of-two scales on the caption rows; the gap rows stay zero
    codes = torch.randint(-4, 5, (rows, D), generator=g, device=DEV).float().to(torch.float8_e4m3fn)
    gal.slots.view(torch.uint8)[keep] = codes.view(torch.uint8)
    gal.scales[keep] = torch.exp2(torch.randint(-1, 2, (rows,), generator=g, device=DEV).float())
    qc = torch.randint(-4, 5, (Nq, D), generator=g, device=DEV).float().to(torch.float8_e4m3fn).view(torch.uint8)
    qs = torch.exp2(torch.randint(-1, 2, (Nq,), generator=g, device=DEV).float())
    ref = _fp64(qc, qs, gal, T)
    for d in (0, 1):
        got = _raw(qc, qs, gal, T, d).double()
        assert torch.equal(got, ref[d][0]), (d, (got - ref[d][0]).abs().max().item())


# ----------------------------------------------------------------------------------------------------------------
# C. scores against fp64
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ci", range(len(_CASES)))
@pytest.mark.parametrize("direction", [0, 1])
@pytest.mark.parametrize("T", _TEMPS)
def test_scores_match_fp64(ci, direction, T):
    q, gal, ref = _case(ci)
    s, A, B, K = ref[T][direction]
    Nq, D = q.shape
    print(f"\nfp8 ragged case {ci} dir {direction}: path {_label(*_path(Nq, gal.n_slots, D, direction))}")
    assert _label(*_path(Nq, gal.n_slots, D, 0)) == _CASES[ci][4]
    tol = _tolerance(D, A, B, K)
    got = R._scores_ragged(q, gal, T, direction).double()
    err = (got - s).abs()
    worst = (err / tol).max().item()
    print(f"n_cap {len(gal)} slots {gal.n_slots} T {T} worst err/tol {worst:.3f}")
    assert torch.isfinite(got).all()
    assert (err <= tol).all(), worst
    k = min(10, len(gal))
    ts, ti = R.retrieve_topk(q, gal, T, k, direction)
    order = torch.from_numpy(np.argsort(-got.cpu().numpy(), kind="stable")[:k]).to(DEV)
    assert torch.equal(ti.long(), order) and torch.equal(ts.double(), got[order])


# ----------------------------------------------------------------------------------------------------------------
# D. direction 0 against Fp8Gallery
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("Nq,dtype", [(77, torch.bfloat16), (300, torch.float32)])
def test_direction_0_equals_fp8_gallery_per_caption(Nq, dtype):
    D, T = 256, 0.07
    lens = np.concatenate([[1, 256, 77, 8, 33], _lengths("cfg3", 40, 81)])
    caps = _captions(lens, D, 82, dtype)
    q = torch.randn(Nq, D, generator=torch.Generator(device=DEV).manual_seed(83), device=DEV)
    gal = R.RaggedGallery.from_list(caps, fp8=True)
    got = R._scores_ragged(q, gal, T, 0)
    want = torch.cat([R._scores_fp8(q, R.quantize_gallery(c[None]), T, 0) for c in caps])
    assert torch.equal(got, want), (got - want).abs().max().item()


# ----------------------------------------------------------------------------------------------------------------
# E. robustness
# ----------------------------------------------------------------------------------------------------------------
def test_nonfinite_caption_row_and_query_token():
    D = 128
    caps = _captions(_lengths("cfg3", 300, 91), D, 92, torch.float32)
    caps[7] = caps[7].clone()
    caps[7][3, 5] = float("nan")
    caps[150] = caps[150].clone()
    caps[150][-1, 0] = float("inf")
    gal = R.RaggedGallery.from_list(caps, fp8=True)
    q = torch.randn(100, D, generator=torch.Generator(device=DEV).manual_seed(93), device=DEV)
    bad = torch.zeros(len(caps), dtype=torch.bool, device=DEV)
    bad[7] = bad[150] = True
    for d in (0, 1):
        s = R._scores_ragged(q, gal, 1.5, d)
        assert torch.isnan(s[bad]).all() and torch.isfinite(s[~bad]).all(), d
    q[42, 9] = float("inf")
    for d in (0, 1):
        assert torch.isnan(R._scores_ragged(q, gal, 1.5, d)).all(), d


def test_deterministic_and_position_independent():
    D, Nq = 256, 300
    lens = _lengths("cfg3", 500, 51)
    caps = _captions(lens, D, 52)
    q = torch.randn(Nq, D, generator=torch.Generator(device=DEV).manual_seed(53), device=DEV).bfloat16()
    gal = R.RaggedGallery.from_list(caps, fp8=True)
    for prefix in (np.array([1]), np.array([17, 200]), _lengths("cfg3", 37, 54)):
        pre = _captions(prefix, D, 55)
        shifted = R.RaggedGallery.from_list(pre + caps, fp8=True)
        joined = R.RaggedGallery.cat([R.RaggedGallery.from_list(pre, fp8=True), gal])
        for d in (0, 1):
            s = R._scores_ragged(q, gal, 0.07, d)
            assert torch.equal(R._scores_ragged(q, gal, 0.07, d).view(torch.int32), s.view(torch.int32))
            assert torch.equal(R._scores_ragged(q, shifted, 0.07, d)[len(pre):], s), (d, prefix.tolist())
            assert torch.equal(R._scores_ragged(q, joined, 0.07, d)[len(pre):], s), (d, prefix.tolist())


def test_no_host_synchronisation_and_no_gallery_sized_temporary():
    D = 512
    gal = R.RaggedGallery.from_list(_captions(_lengths("cfg3", 3000, 61), D, 62), fp8=True)
    q = torch.randn(256, D, device=DEV).bfloat16()
    T = torch.tensor(0.07, device=DEV)
    ref = {d: R.retrieve_topk(q, gal, T, 10, d) for d in (0, 1)}          # workspaces allocated
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        out = {d: R.retrieve_topk(q, gal, T, 10, d) for d in (0, 1)}
    finally:
        torch.cuda.set_sync_debug_mode("default")
    for d in (0, 1):
        assert torch.equal(out[d][1], ref[d][1]) and torch.equal(out[d][0], ref[d][0])
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        R.retrieve_topk(q, gal, T, 10, d)
        torch.cuda.synchronize()
        extra = torch.cuda.max_memory_allocated() - base
        assert extra < gal.nbytes / 100, (d, extra, gal.nbytes)
    n_rows = gal.n_slots * SLOT
    assert gal.nbytes == n_rows * D + 4 * n_rows + 4 * gal.meta.numel() + 4 * gal.cap_info.numel()


# ----------------------------------------------------------------------------------------------------------------
# F. against the bf16 ragged gallery
# ----------------------------------------------------------------------------------------------------------------
def test_planted_order_agrees_with_bf16():
    D, Nq, T = 512, 64, 1.5
    g = torch.Generator(device=DEV).manual_seed(71)
    u = torch.nn.functional.normalize(torch.randn(D, generator=g, device=DEV), dim=0)
    q = torch.nn.functional.normalize(u + 0.5 * torch.randn(Nq, D, generator=g, device=DEV) / D ** 0.5, dim=1)
    lens = _lengths("cfg3", 1500, 72)
    caps = [c.float() for c in _captions(lens, D, 73)]
    levels = [0.9, 0.8, 0.7, 0.6, 0.5, 0.4]
    planted = [1400, 3, 777, 250, 1001, 60]                      # in descending order of level
    for i, c in zip(planted, levels):
        noise = torch.nn.functional.normalize(torch.randn(int(lens[i]), D, generator=g, device=DEV), dim=1)
        caps[i] = torch.nn.functional.normalize(c * u + (1 - c * c) ** 0.5 * noise, dim=1)
    g8 = R.RaggedGallery.from_list(caps, fp8=True)
    g16 = R.RaggedGallery.from_list(caps)
    qc, qs = _quant(q)
    ref8 = _fp64(qc, qs, g8, T)
    qb = q.bfloat16().double()
    cid = _segments(g16)
    keep = cid < len(caps)
    e16 = g16.slots[keep].double() @ qb.T / T
    lens_t = torch.from_numpy(lens.astype(np.int64)).to(DEV)
    ref16 = {0: torch.full((len(caps), Nq), -float("inf"), dtype=torch.float64, device=DEV).scatter_reduce_(
                 0, cid[keep][:, None].expand_as(e16), e16, "amax").mean(1),
             1: torch.zeros(len(caps), dtype=torch.float64, device=DEV).index_add_(0, cid[keep], e16.amax(1)) / lens_t}
    for d in (0, 1):
        r8, r16 = ref8[d][0], ref16[d]
        qerr = (r8 - r16).abs()                                  # the quantization error, per caption
        margin = 2 * qerr.max() + 1e-3
        rest = torch.ones(len(caps), dtype=torch.bool, device=DEV)
        rest[planted] = False
        for r in (r8, r16):                                      # premise: the planted levels are further apart
            pr = torch.cat([r[planted], r[rest].max()[None]])
            assert ((pr[:-1] - pr[1:]) > margin).all(), (d, pr.tolist(), margin.item())
        k = len(planted)
        _, i8 = R.retrieve_topk(q, g8, T, k, d)
        _, i16 = R.retrieve_topk(q, g16, T, k, d)
        assert i8.tolist() == i16.tolist() == planted, d
        print(f"\ndirection {d}: worst quantization error {qerr.max().item():.2e}")


# ----------------------------------------------------------------------------------------------------------------
# G. gallery-sharded top-k
# ----------------------------------------------------------------------------------------------------------------
def test_sharded_single_rank_matches_retrieve_topk():
    from triad_b200.dist import sharded_retrieve_topk
    D = 128
    caps = _captions(_lengths("cfg3", 700, 71), D, 72)
    caps[650] = caps[17]                                                   # a tie
    q = torch.nn.functional.normalize(torch.randn(77, D, device=DEV), dim=1).bfloat16()
    gal = R.RaggedGallery.from_list(caps, fp8=True)
    shard = R.RaggedGallery.from_list(caps[300:], fp8=True)
    for d in (0, 1):
        s, ids = sharded_retrieve_topk(q, gal, 1.5, 12, 0, direction=d)
        s0, i0 = R.retrieve_topk(q, gal, 1.5, 12, d)
        assert torch.equal(ids, i0.long()) and torch.equal(s, s0)
        assert torch.equal(R._scores_ragged(q, shard, 1.5, d), R._scores_ragged(q, gal, 1.5, d)[300:])
        s1, i1 = sharded_retrieve_topk(q, shard, 1.5, 12, 300, direction=d)
        assert (i1 >= 300).all()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least 2 GPUs")
def test_sharded_fp8_ragged_retrieval_under_nccl():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", "29523", os.path.join("tools", "sharded_retrieval_check.py"),
           "--ragged", "--fp8"]
    r = subprocess.run(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    assert "SHARDED_RETRIEVAL_OK" in r.stdout
