"""GPU tier: retrieval on an e4m3 gallery (``Fp8Gallery``, ``triad_quantize_e4m3``, ``triad_retrieve_scores_e4m3``).

Contract.  A row x[0..D) is quantized as s = fp32(amax / 448), c = e4m3_rn_satfinite(fp32(x / s)) (c = 0 when s == 0;
s = NaN when the row holds an inf or a NaN).  The score of image n for a query with codes cq, token scales sq is
    score_n = sum_a fp32(m_a t_a),  m_a = max_p fp32(sg_p acc_ap),  acc_ap = sum_k cq_ak cg_pk  (tensor cores),
    t_a = fp32(fp32(sq_a fp32(1/Nq)) fp32(1/T)),
i.e. exact arithmetic on the quantized values up to the accumulator and the fp32 roundings named here.

A. The quantizer, bit for bit against torch.clamp(x / s, -448, 448).to(float8_e4m3fn) on the CPU (fp32 and bf16
   inputs; Gaussian, unit-norm and wide-range rows, all-zero / underflowing / single non-zero / -0.0 rows), ``put`` at
   an offset, and slicing: quantizing a slice of a gallery gives that slice of the quantized gallery.
B1. Exact layout probe: small-integer codes, power-of-two scales, Nq and T.  Every partial sum is an integer far
   below 2^24 times a power of two, so every operation is exact and the scores must equal fp64 bit for bit, whatever
   the accumulator does with bits it never needs.  Any k-block, column-scale or row indexing error shows here.
B2. Accumulator probe: acc = 256*256 + 127 * 2^-j (one 2^16 product and 127 products 2^-j across all four k-blocks
   of D = 128).  A full fp32 accumulator is exact up to j = 7 (24 significant bits); one that keeps b bits aligned
   to the largest product is exact up to j = b - 17.  The number of bits found (B2 asserts the exact cases form a
   prefix, as such a model implies) sets the accumulator term of C's tolerance.  On a B200 (1000 W) the probe is exact
   up to j = 7 and not beyond: the full fp32 model holds, b = 24.
C. Scores against fp64 of the dequantized operands, per image, on every path a one-query fp8 retrieval takes (tc1 /
   tc2, default / retrieval / chunk-synchronous tile order, with and without 256-patch sub-tiles, D 128 to 512).
   With bits b from B2 (24 for a full fp32 accumulator), per score
       tol_n = (1 + 2^-6) (D 2^-(b-1) B_n + (Nq + 8) 2^-23 A_n),
       A_n = mean_a max_p |e_ap|,  B_n = mean_a max_p sq_a sg_p sum_k |cq_ak cg_pk| / T
   (D accumulation steps of at most 2^-(b-1) of the sum of magnitudes each; the products by sg, sq, 1/Nq, 1/T and t_a
   and the fp32 sum over Nq tokens take at most (Nq + 8) roundings of 2^-24).  Planted images (every patch at cosine
   c with a query token, graded c) must be more than 10x the largest tolerance apart — each case asserts it — and two
   exact copies in different tile chunks must score bit-equal and rank by id.  Top-k is exact on the planted images
   and certified in the random tail.
D. Against the bf16 path: on a planted gallery, the planted ids and their order agree; the premise gap covers the
   quantization error, |fp64 score of the dequantized gallery - fp64 score of the bf16 one| per item.  The top-10
   overlap on a random gallery is printed, not asserted.
E. A non-finite gallery row gives a NaN score for its image only; two runs are bit-identical; the call allocates no
   gallery-sized temporary; ``nbytes``.
F. Gallery-sharded fp8 top-k under NCCL (>= 2 GPUs, skipped otherwise).
"""
import math
import os
import subprocess
import sys

import pytest
import torch

from triad_b200 import _lib, ops, retrieval as R
from triad_b200._lib import check

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_SMS = torch.cuda.get_device_properties(0).multi_processor_count if torch.cuda.is_available() else 148
_MiB = 1 << 20
DEV = "cuda"


# ----------------------------------------------------------------------------------------------------------------
# references
# ----------------------------------------------------------------------------------------------------------------
def _quant_ref(x: torch.Tensor):
    """The contract on the CPU: (codes uint8 [..., D], scales fp32 [...])."""
    x = x.detach().cpu().float()
    amax = x.abs().amax(dim=-1)
    s = amax / 448.0
    s = torch.where(torch.isfinite(amax), s, torch.full_like(s, float("nan")))
    ok = (s > 0)[..., None]
    safe = torch.where(ok, s[..., None], torch.ones_like(s[..., None]))
    c = torch.clamp(x / safe, -448, 448).to(torch.float8_e4m3fn).view(torch.uint8)
    c = torch.where(ok, c, torch.zeros_like(c))
    return c, s


def _quant_gpu(x: torch.Tensor):
    D = x.shape[-1]
    codes = torch.empty(x.shape, dtype=torch.uint8, device=x.device)
    scales = torch.empty(x.shape[:-1], dtype=torch.float32, device=x.device)
    R._quantize_rows(x, codes, scales)
    return codes, scales


def _deq(codes_u8: torch.Tensor, scales: torch.Tensor) -> torch.Tensor:
    return codes_u8.view(torch.float8_e4m3fn).double() * scales.double()[..., None]


def _fp64_scores(qc, qs, gc, gs, T):
    """(score, A, B) per image in fp64, the operands dequantized exactly."""
    q = _deq(qc, qs)                                      # [Nq, D]
    qa = qc.view(torch.float8_e4m3fn).double().abs()
    n, Nv, D = gc.shape
    chunk = max(1, min(4096, (1 << 28) // (Nv * max(D, q.shape[0]) * 8)))
    out, A, B = [], [], []
    for i in range(0, n, chunk):
        c = gc[i:i + chunk]
        g = _deq(c, gs[i:i + chunk])                      # [b, Nv, D]
        e = torch.einsum("ad,bpd->bap", q, g) / T
        out.append(e.amax(dim=2).mean(dim=1))
        A.append(e.abs().amax(dim=2).mean(dim=1))
        mag = torch.einsum("ad,bpd->bap", qa, c.view(torch.float8_e4m3fn).double().abs())
        mag = mag * qs.double()[None, :, None] * gs[i:i + chunk].double()[:, None, :] / T
        B.append(mag.amax(dim=2).mean(dim=1))
    return torch.cat(out), torch.cat(A), torch.cat(B)


def _scores_raw(qc, qs, gc, gs, T):
    lib = _lib.load()
    Nq, D = qc.shape
    n, Nv = gs.shape
    Tt = ops.temperature_tensor(T, qc.device)
    out = torch.empty(n, dtype=torch.float32, device=qc.device)
    nws = lib.triad_retrieve_e4m3_workspace_bytes(Nq, n, Nv, D)
    ws = torch.empty(nws, dtype=torch.uint8, device=qc.device)
    check(lib.triad_retrieve_scores_e4m3(qc.data_ptr(), qs.data_ptr(), Nq, gc.data_ptr(), gs.data_ptr(), n, Nv, D,
                                         Tt.data_ptr(), out.data_ptr(), ws.data_ptr(), nws, ops._stream(qc.device)),
          "triad_retrieve_scores_e4m3")
    return out


# ----------------------------------------------------------------------------------------------------------------
# A. quantizer
# ----------------------------------------------------------------------------------------------------------------
def _quant_inputs(D, g):
    gauss = torch.randn(64, D, generator=g)
    unit = torch.nn.functional.normalize(torch.randn(64, D, generator=g), dim=1)
    e = torch.randint(-20, 11, (64, D), generator=g).float()
    wide = torch.sign(torch.randn(64, D, generator=g)) * torch.exp2(e)             # 2^-20 .. 2^10 inside a row
    rowwide = torch.randn(31, D, generator=g) * torch.exp2(torch.arange(-20, 11).float())[:, None]
    edge = torch.zeros(6, D)
    edge[1, 3] = 1e-45                                     # amax / 448 underflows: s == 0
    edge[2, 5] = -3.0                                      # a single non-zero
    edge[3] = -0.0                                         # all -0.0: s == 0
    edge[4] = torch.randn(D, generator=g)
    edge[4, ::3] = -0.0                                    # -0.0 elements in a live row keep their sign
    edge[5, :] = 2.0 ** -140                               # subnormal fp32 amax, s a subnormal > 0
    return torch.cat([gauss, unit, wide, rowwide, edge])


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("D", [16, 128, 512])
def test_quantizer_bit_exact(dtype, D):
    g = torch.Generator().manual_seed(D)
    x = _quant_inputs(D, g).to(dtype)
    c_ref, s_ref = _quant_ref(x)
    c, s = _quant_gpu(x.to(DEV))
    assert torch.equal(s.cpu().view(torch.int32), s_ref.view(torch.int32))
    assert torch.equal(c.cpu(), c_ref)
    # the premises: subnormal codes, zero scales and -0.0 codes occur
    assert ((c_ref & 0x78) == 0).logical_and((c_ref & 0x07) != 0).any()
    assert (s_ref == 0).sum() >= 2 and (c_ref == 0x80).any()


def test_quantizer_nonfinite_rows_get_nan_scales():
    x = torch.randn(4, 256)
    x[1, 7] = float("inf")
    x[2, 9] = float("nan")
    x[3, 0] = float("-inf")
    c, s = _quant_gpu(x.to(DEV))
    s = s.cpu()
    assert torch.isfinite(s[0]) and torch.isnan(s[1:]).all()


def test_put_at_offset_and_slices():
    g = torch.Generator(device=DEV).manual_seed(3)
    feats = torch.randn(10, 37, 256, generator=g, device=DEV).bfloat16()
    full = R.quantize_gallery(feats)
    c_ref, s_ref = _quant_ref(feats)
    assert torch.equal(full.codes.view(torch.uint8).cpu(), c_ref)
    assert torch.equal(full.scales.cpu().view(torch.int32), s_ref.view(torch.int32))
    part = R.quantize_gallery(feats[3:8])
    assert torch.equal(part.codes.view(torch.uint8), full.codes[3:8].view(torch.uint8))
    assert torch.equal(part.scales, full.scales[3:8])
    sl = full[3:8]
    assert torch.equal(sl.codes.view(torch.uint8), part.codes.view(torch.uint8))
    gal = R.Fp8Gallery.empty(10, 37, 256, device=DEV)
    gal.codes.view(torch.uint8).fill_(0x5a)
    gal.scales.fill_(7.0)
    gal.put(4, feats[4:6])
    assert torch.equal(gal.codes[4:6].view(torch.uint8), full.codes[4:6].view(torch.uint8))
    assert torch.equal(gal.scales[4:6], full.scales[4:6])
    assert (gal.codes[:4].view(torch.uint8) == 0x5a).all() and (gal.codes[6:].view(torch.uint8) == 0x5a).all()
    assert (gal.scales[:4] == 7.0).all() and (gal.scales[6:] == 7.0).all()


# ----------------------------------------------------------------------------------------------------------------
# B1. exact layout probe
# ----------------------------------------------------------------------------------------------------------------
def _int_codes(shape, lo, hi, g):
    v = torch.randint(lo, hi + 1, shape, generator=g, device=DEV).float()
    return v.to(torch.float8_e4m3fn).view(torch.uint8)


@pytest.mark.parametrize("Nq,n,Nv,D,T", [(1, 37, 13, 128, 0.5), (64, 50, 256, 512, 2.0), (128, 40, 300, 256, 1.0),
                                         (256, 30, 257, 512, 0.25), (256, 60, 1, 384, 4.0)])
def test_exact_layout_probe(Nq, n, Nv, D, T):
    g = torch.Generator(device=DEV).manual_seed(Nq * 7 + D)
    qc = _int_codes((Nq, D), -4, 4, g)
    gc = _int_codes((n, Nv, D), -4, 4, g)
    qs = torch.exp2(torch.randint(-1, 2, (Nq,), generator=g, device=DEV).float())
    gs = torch.exp2(torch.randint(-1, 2, (n, Nv), generator=g, device=DEV).float())
    ref, _, _ = _fp64_scores(qc, qs, gc, gs, T)
    # premise: every fp32 partial sum is exact (integer multiples of 2^-e below 2^24 2^-e)
    q = qc.view(torch.float8_e4m3fn).double()
    unit = 0.25 / (Nq * T)                # every term m_a t_a is an integer multiple of this (sg, sq in {1/2, 1, 2})
    for i in range(0, n, 16):
        acc = torch.einsum("ad,bpd->bap", q, gc[i:i + 16].view(torch.float8_e4m3fn).double())
        assert acc.abs().max() < 2 ** 16
        terms = (acc * gs[i:i + 16].double()[:, None, :]).amax(dim=2) * qs.double() / Nq / T
        assert ((terms.abs().sum(dim=1) / unit) < 2 ** 24).all()
    out = _scores_raw(qc, qs, gc, gs, T)
    assert torch.equal(out.double(), ref), (out.double() - ref).abs().max()


# ----------------------------------------------------------------------------------------------------------------
# B2. accumulator probe
# ----------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="session")
def acc_bits():
    D, J = 128, 10                        # 2^-9 is the smallest e4m3 subnormal
    qv = torch.zeros(J, D, device=DEV)
    gv = torch.zeros(J, 1, D, device=DEV)
    for j in range(J):
        qv[j, 0], gv[j, 0, 0] = 256.0, 256.0
        qv[j, 1:] = 2.0 ** -j
        gv[j, 0, 1:] = 1.0
    exact = []
    for j in range(J):
        qc = qv[j:j + 1].to(torch.float8_e4m3fn).view(torch.uint8)
        gc = gv[j:j + 1].to(torch.float8_e4m3fn).view(torch.uint8)
        ones = torch.ones(1, device=DEV)
        s = _scores_raw(qc, ones, gc, ones.reshape(1, 1), 1.0).item()
        exact.append(s == 65536.0 + 127 * 2.0 ** -j)
    jmax = -1
    while jmax + 1 < J and exact[jmax + 1]:
        jmax += 1
    return {"exact": exact, "bits": 17 + jmax}


def test_accumulator_probe(acc_bits):
    exact = acc_bits["exact"]
    k = sum(exact)
    print(f"\nfp8 accumulator probe: exact for j < {k} of {len(exact)}: {acc_bits['bits']} significant bits "
          f"({'a full fp32 accumulator' if acc_bits['bits'] >= 24 else 'a truncating accumulator'})")
    assert exact == [True] * k + [False] * (len(exact) - k), exact    # a prefix, as either model implies
    assert acc_bits["bits"] >= 14


def _acc_rel(acc_bits):
    return 2.0 ** -(min(acc_bits["bits"], 24) - 1)


# ----------------------------------------------------------------------------------------------------------------
# C. scores and top-k against fp64 on every path
# ----------------------------------------------------------------------------------------------------------------
def _fp8_path(Nq, n, Nv, D, sms=_SMS):
    """(kernel, tile order, C, sub-tiles): launch_maxmean_tc's e4m3 path with the e4m3 image size Nv*D."""
    cta = 1 if Nq <= 128 else 2
    n_m = -(-Nq // (128 * cta))
    img = Nv * D
    clusters = sms // cta
    order, C = "default", n
    if n * img > 48 * _MiB:
        c16 = max(1, 16 * _MiB // img)
        if n_m * c16 >= 4 * clusters:
            order, C = "sync", min(c16, n)
        else:
            order, C = "retrieval", min(max(1, min(64, 48 * _MiB // (clusters * img))), n)
    return f"tc{cta}", order, C, Nv > 256


CASES = [  # Nq, n_img, Nv, D
    (77, 300, 1024, 512),      # tc1, retrieval order C = 1, sub-tiles (cfg 5 text, smaller gallery)
    (250, 200, 1024, 512),     # tc2, retrieval order C = 1, sub-tiles (cfg 5 audio)
    (77, 1700, 64, 512),       # tc1, retrieval order C = 10
    (250, 700, 1024, 128),     # tc2, retrieval order C = 5, sub-tiles
    (256, 1700, 64, 512),      # tc2, chunk-synchronous order
    (1, 40000, 13, 128),       # tc1, chunk-synchronous order, one token
    (128, 500, 257, 256),      # tc1, default order, a 1-patch last sub-tile
    (129, 500, 256, 256),      # tc2, default order
    (256, 300, 255, 128),      # tc2, default order
    (1, 1000, 1, 512),         # one patch
]


def test_cases_cover_every_fp8_path():
    paths = [_fp8_path(*c) for c in CASES]
    kinds = {p[0] for p in paths}
    orders = {(p[0], p[1]) for p in paths}
    assert kinds == {"tc1", "tc2"}
    assert {("tc1", "default"), ("tc2", "default"), ("tc1", "retrieval"), ("tc2", "retrieval"), ("tc1", "sync"),
            ("tc2", "sync")} <= orders
    Cs = {p[2] for p in paths if p[1] == "retrieval"}
    assert 1 in Cs and max(Cs) > 1
    assert {p[3] for p in paths} == {True, False}
    assert {c[3] for c in CASES} >= {128, 256, 512}
    assert {c[0] for c in CASES} >= {1, 77, 128, 129, 250, 256}
    assert {c[2] for c in CASES} >= {1, 13, 255, 256, 257, 1024}


LEVELS = [0.95, 0.9, 0.85, 0.8, 0.75, 0.7, 0.65, 0.6]


def _planted_gallery(Nq, n, Nv, D, seed):
    """(q [Nq, D] fp32, feats [n, Nv, D] bf16, planted ids in level order, copy pairs)."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    q = torch.nn.functional.normalize(torch.randn(Nq, D, generator=g, device=DEV), dim=1)
    feats = torch.empty(n, Nv, D, dtype=torch.bfloat16, device=DEV)
    step = max(1, (256 * _MiB) // (Nv * D * 4))
    for i in range(0, n, step):
        b = min(step, n - i)
        feats[i:i + b] = torch.nn.functional.normalize(torch.randn(b, Nv, D, generator=g, device=DEV), dim=2).bfloat16()
    C = _fp8_path(Nq, n, Nv, D)[2]
    cands = [0, n - 1, min(C, n - 1), max(0, C - 1), 4095, 4096, n // 2, n // 3, 1, n - 2]
    ids = []
    for c in cands:
        if 0 <= c < n and c not in ids:
            ids.append(c)
    ids = ids[:len(LEVELS)]
    tok = q[torch.arange(Nv, device=DEV) % Nq]                                   # [Nv, D]
    for lvl, j in zip(LEVELS, ids):
        noise = torch.randn(Nv, D, generator=g, device=DEV)
        noise = noise - (noise * tok).sum(1, keepdim=True) * tok
        noise = torch.nn.functional.normalize(noise, dim=1)
        feats[j] = (lvl * tok + math.sqrt(1 - lvl * lvl) * noise).bfloat16()
    # two copies: the last planted image duplicated at another id (far away: another chunk)
    pairs = []
    if n >= 4 and len(ids) >= 2:
        src = ids[0]
        dst = next(c for c in (n - 3, n // 2 + 1, 2) if c not in ids and 0 <= c < n)
        feats[dst] = feats[src]
        pairs.append((src, dst))
    return q, feats, ids, pairs


_GAL_CACHE = {}


def _case_data(ci, acc_bits):
    if ci in _GAL_CACHE:
        return _GAL_CACHE[ci]
    _GAL_CACHE.clear()
    torch.cuda.empty_cache()
    Nq, n, Nv, D = CASES[ci]
    T = 1.5
    q, feats, planted, pairs = _planted_gallery(Nq, n, Nv, D, seed=100 + ci)
    gal = R.quantize_gallery(feats)
    del feats
    qc, qs = _quant_gpu(q)
    ref, A, B = _fp64_scores(qc, qs, gal.codes.view(torch.uint8), gal.scales, T)
    tol = (1 + 2 ** -6) * (D * _acc_rel(acc_bits) * B + (Nq + 8) * 2.0 ** -23 * A)
    d = dict(q=q, gal=gal, T=T, ref=ref, tol=tol, planted=planted, pairs=pairs)
    _GAL_CACHE[ci] = d
    return d


@pytest.mark.parametrize("ci", range(len(CASES)), ids=[f"Nq{c[0]}-n{c[1]}-Nv{c[2]}-D{c[3]}" for c in CASES])
def test_scores_and_topk_match_fp64(ci, acc_bits):
    d = _case_data(ci, acc_bits)
    ref, tol, planted = d["ref"], d["tol"], d["planted"]
    print(f"\n{CASES[ci]} path {_fp8_path(*CASES[ci])}")
    # premise: planted fp64 scores more than 10x the largest tolerance apart
    pr = ref[planted]
    gaps = (pr[:-1] - pr[1:])
    assert (gaps > 10 * tol.max()).all(), (gaps.min().item(), tol.max().item())
    qc, qs = _quant_gpu(d["q"])
    s = _scores_raw(qc, qs, d["gal"].codes.view(torch.uint8), d["gal"].scales, d["T"])
    err = (s.double() - ref).abs()
    assert torch.isfinite(s).all()
    assert (err <= tol).all(), f"worst err/tol {(err / tol).max().item():.3f}"
    print(f"worst err/tol {(err / tol).max().item():.3e}, max tol {tol.max().item():.3e}")
    for a, b in d["pairs"]:
        assert s[a].view(torch.int32) == s[b].view(torch.int32)
    k = min(20, ref.numel())
    ts, ti = R.retrieve_topk(d["q"], d["gal"], d["T"], k)
    ti = ti.long()
    assert torch.equal(ts, s[ti])                                              # the kernel's own scores, bit for bit
    want = sorted(planted + [b for _, b in d["pairs"]], key=lambda j: (-ref[j].item(), j))[:k]
    assert ti[:len(want)].tolist() == want                                     # exact on the planted images
    # certified tail: nothing left out could beat what was returned
    mask = torch.ones_like(ref, dtype=torch.bool)
    mask[ti] = False
    if mask.any():
        assert (ref[ti] + tol[ti]).min() >= (ref[mask] - tol[mask]).max()


# ----------------------------------------------------------------------------------------------------------------
# D. against the bf16 path
# ----------------------------------------------------------------------------------------------------------------
def test_planted_order_agrees_with_bf16(acc_bits):
    Nq, n, Nv, D, T = 77, 600, 1024, 512, 1.5
    q, feats, planted, pairs = _planted_gallery(Nq, n, Nv, D, seed=7)
    gal = R.quantize_gallery(feats)
    qc, qs = _quant_gpu(q)
    ref8, _, _ = _fp64_scores(qc, qs, gal.codes.view(torch.uint8), gal.scales, T)
    qb = q.bfloat16()
    ref16 = torch.cat([(torch.einsum("ad,bpd->bap", qb.double(), feats[i:i + 64].double()) / T).amax(2).mean(1)
                       for i in range(0, n, 64)])
    qerr = (ref8 - ref16).abs()                                               # the quantization error, per item
    pr8 = ref8[planted]
    pr16 = ref16[planted]
    margin = 2 * qerr[planted].max() + 1e-3
    assert ((pr8[:-1] - pr8[1:]) > margin).all() and ((pr16[:-1] - pr16[1:]) > margin).all()
    k = 10
    _, i8 = R.retrieve_topk(q, gal, T, k)
    _, i16 = R.retrieve_topk(qb, feats, T, k)
    want = sorted(planted + [b for _, b in pairs], key=lambda j: (-ref16[j].item(), j))
    assert i8[:len(want)].tolist() == i16[:len(want)].tolist() == want
    # random gallery: report the overlap of the two top-10s
    g = torch.Generator(device=DEV).manual_seed(11)
    rnd = torch.nn.functional.normalize(torch.randn(n, Nv, D, generator=g, device=DEV), dim=2).bfloat16()
    _, a = R.retrieve_topk(qb, rnd, T, k)
    _, b = R.retrieve_topk(q, R.quantize_gallery(rnd), T, k)
    print(f"\nrandom gallery {n} x {Nv} x {D}, Nq {Nq}: top-10 overlap fp8 vs bf16 "
          f"{len(set(a.tolist()) & set(b.tolist()))}/10, worst planted quantization error {qerr[planted].max().item():.2e}")


# ----------------------------------------------------------------------------------------------------------------
# E. robustness and behaviour
# ----------------------------------------------------------------------------------------------------------------
def test_nonfinite_gallery_row_gives_nan_for_that_image_only():
    g = torch.Generator(device=DEV).manual_seed(9)
    feats = torch.nn.functional.normalize(torch.randn(40, 300, 256, generator=g, device=DEV), dim=2)
    feats[5, 17, 3] = float("nan")
    feats[21, 299, 0] = float("inf")
    gal = R.quantize_gallery(feats)
    q = torch.randn(77, 256, generator=g, device=DEV)
    qc, qs = _quant_gpu(q)
    s = _scores_raw(qc, qs, gal.codes.view(torch.uint8), gal.scales, 1.5)
    bad = torch.zeros(40, dtype=torch.bool, device=DEV)
    bad[5] = bad[21] = True
    assert torch.isnan(s[bad]).all() and torch.isfinite(s[~bad]).all()


def test_bit_identical_runs_and_no_gallery_sized_temporary():
    g = torch.Generator(device=DEV).manual_seed(12)
    feats = torch.nn.functional.normalize(torch.randn(400, 1024, 512, generator=g, device=DEV), dim=2).bfloat16()
    gal = R.quantize_gallery(feats)
    del feats
    q = torch.randn(250, 512, generator=g, device=DEV).bfloat16()
    s1, i1 = R.retrieve_topk(q, gal, 1.5, 10)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    s2, i2 = R.retrieve_topk(q, gal, 1.5, 10)
    torch.cuda.synchronize()
    extra = torch.cuda.max_memory_allocated() - base
    assert torch.equal(s1.view(torch.int32), s2.view(torch.int32)) and torch.equal(i1, i2)
    assert extra < gal.nbytes / 100, (extra, gal.nbytes)
    assert gal.nbytes == 400 * 1024 * 512 + 4 * 400 * 1024
    assert gal.nbytes == gal.codes.numel() * gal.codes.element_size() + gal.scales.numel() * 4


# ----------------------------------------------------------------------------------------------------------------
# F. gallery-sharded fp8 top-k
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least 2 GPUs")
def test_sharded_fp8_retrieval_under_nccl():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", "29519", os.path.join("tools", "sharded_retrieval_check.py"),
           "--fp8"]
    r = subprocess.run(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    assert "SHARDED_RETRIEVAL_OK" in r.stdout


def test_sharded_fp8_single_rank_matches_retrieve_topk():
    from triad_b200.dist import sharded_retrieve_topk
    g = torch.Generator(device=DEV).manual_seed(5)
    q = torch.nn.functional.normalize(torch.randn(77, 128, generator=g, device=DEV), dim=1).bfloat16()
    feats = torch.nn.functional.normalize(torch.randn(300, 64, 128, generator=g, device=DEV), dim=2).bfloat16()
    feats[250] = feats[17]
    gal = R.quantize_gallery(feats)
    s, ids = sharded_retrieve_topk(q, gal, 1.5, 12, 0)
    s0, i0 = R.retrieve_topk(q, gal, 1.5, 12)
    assert torch.equal(ids, i0.long()) and torch.equal(s, s0)
    # a shard with an id offset scores exactly the slice of the whole gallery
    s1, i1 = sharded_retrieve_topk(q, gal[100:300], 1.5, 12, 100)
    s_all = R._scores_fp8(q, gal, 1.5, 0)
    assert torch.equal(R._scores_fp8(q, gal[100:300], 1.5, 0), s_all[100:300])
    assert (i1 >= 100).all()
